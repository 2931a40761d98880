// solver.cu -- host orchestration behind the C ABI (include/tlsq_b200.h): handle, NCCL plumbing (dlopen, so the
// library loads on machines without NCCL or a GPU), and the three solver loops
//   rpca_core        inexact ALM               (src/robustPCA.jl:156-239)
//   rpca_ga_core     Grassmann averages        (src/robustPCA.jl:255-306)
//   lowrankfilter    rpca on an implicit Hankel embedding + anti-diagonal averaging (:119-128)
// There is no CPU fallback anywhere in this file: every path launches the sm_100a kernels or fails.
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <vector>

#include "../../include/tlsq_b200.h"
#include "kernels.h"

using namespace tlsq;

// ------------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int set_err(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CK(expr)                                                                                         \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess) {                                                                         \
            int _code = (_e == cudaErrorMemoryAllocation) ? TLSQ_ERR_NOMEM : TLSQ_ERR_CUDA;              \
            return set_err(_code, "CUDA error '%s' at %s:%d (%s)", cudaGetErrorString(_e), __FILE__,     \
                           __LINE__, #expr);                                                             \
        }                                                                                                \
    } while (0)

#define CKR(expr)                                \
    do {                                         \
        int _r = (expr);                         \
        if (_r != TLSQ_OK) return _r;            \
    } while (0)

// ------------------------------------------------------------------------------------------------------
// NCCL through dlopen
// ------------------------------------------------------------------------------------------------------
namespace {
struct NcclId { char internal[128]; };
typedef int (*fn_get_uid)(NcclId*);
typedef int (*fn_init_rank)(void**, int, NcclId, int);
typedef int (*fn_allreduce)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*fn_destroy)(void*);
typedef const char* (*fn_errstr)(int);

struct NcclApi {
    void* lib = nullptr;
    fn_get_uid get_uid = nullptr;
    fn_init_rank init_rank = nullptr;
    fn_allreduce allreduce = nullptr;
    fn_destroy destroy = nullptr;
    fn_errstr errstr = nullptr;
    bool tried = false;
};
NcclApi g_nccl;
constexpr int kNcclFloat64 = 8, kNcclSum = 0, kNcclMax = 2;

int nccl_load() {
    if (g_nccl.lib) return TLSQ_OK;
    if (!g_nccl.tried) {
        g_nccl.tried = true;
        const char* env = getenv("TLSQ_NCCL_LIB");
        const char* cands[] = {env, "libnccl.so.2", "libnccl.so"};
        for (const char* c : cands) {
            if (!c || !*c) continue;
            g_nccl.lib = dlopen(c, RTLD_NOW | RTLD_GLOBAL);
            if (g_nccl.lib) break;
        }
        if (g_nccl.lib) {
            g_nccl.get_uid = (fn_get_uid)dlsym(g_nccl.lib, "ncclGetUniqueId");
            g_nccl.init_rank = (fn_init_rank)dlsym(g_nccl.lib, "ncclCommInitRank");
            g_nccl.allreduce = (fn_allreduce)dlsym(g_nccl.lib, "ncclAllReduce");
            g_nccl.destroy = (fn_destroy)dlsym(g_nccl.lib, "ncclCommDestroy");
            g_nccl.errstr = (fn_errstr)dlsym(g_nccl.lib, "ncclGetErrorString");
            if (!g_nccl.get_uid || !g_nccl.init_rank || !g_nccl.allreduce || !g_nccl.destroy) g_nccl.lib = nullptr;
        }
    }
    if (!g_nccl.lib)
        return set_err(TLSQ_ERR_NCCL, "libnccl.so.2 not loadable (set TLSQ_NCCL_LIB to its path): %s",
                       dlerror() ? dlerror() : "symbols missing");
    return TLSQ_OK;
}
}  // namespace

// ------------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------------
struct tlsq_handle {
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t side = nullptr;          // output pass of the finalisation overlaps the full eigensolver
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_iter = nullptr, ev_d2h = nullptr;
    int64_t launches = 0;
    cudaMemPool_t pool = nullptr;         // private stream-ordered pool (release threshold: keep everything)
    void* comm = nullptr;
    int nranks = 1;
    int rank = 0;
    double* h_pin = nullptr;     // pinned host scratch (64 doubles)
    // optional per-phase device timing (CUDA events on the solve stream)
    bool prof = false;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    struct Span { int phase; cudaEvent_t a, b; };
    std::vector<Span> spans;
    double phase_ms[TLSQ_NUM_PHASES] = {0};
    int64_t phase_calls[TLSQ_NUM_PHASES] = {0};
};

namespace {

// stream-ordered allocations come from the calling handle's PRIVATE memory pool (set by use_device): freed blocks stay
// cached between solves without touching the attributes of the device's default pool, which a co-resident allocator
// (PyTorch) may be using
thread_local cudaMemPool_t t_pool = nullptr;
// set when a solve left the accelerated large-embedding path (rank estimate beyond the 32-column factors, or hankel=true
// with min(M,N) > 512):
// tlsq_rpca_f64 then repeats the solve on the dense device path (rpca_cb_host with the built-in hooks)
thread_local bool t_dense_fallback = false;

struct DevBuf {                  // stream-ordered device allocation, freed on scope exit
    void* p = nullptr;
    cudaStream_t st = nullptr;
    cudaError_t alloc(size_t bytes, cudaStream_t s) {
        st = s;
        if (bytes == 0) bytes = 8;
        if (t_pool) return cudaMallocFromPoolAsync(&p, bytes, t_pool, s);
        return cudaMallocAsync(&p, bytes, s);
    }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
    void release() { if (p) { cudaFreeAsync(p, st); p = nullptr; } }
    ~DevBuf() { release(); }
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
};

cudaEvent_t prof_event(tlsq_handle* h) {
    if (h->ev_used == h->ev_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        h->ev_pool.push_back(e);
    }
    return h->ev_pool[h->ev_used++];
}

struct Phase {                   // RAII span: records start/stop events on the solve stream when profiling is on
    tlsq_handle* h;
    int phase;
    cudaEvent_t a = nullptr;
    Phase(tlsq_handle* hh, int ph) : h(hh), phase(ph) {
        if (h->prof) { a = prof_event(h); cudaEventRecord(a, h->stream); }
    }
    ~Phase() {
        if (h->prof && a) {
            cudaEvent_t b = prof_event(h);
            cudaEventRecord(b, h->stream);
            h->spans.push_back({phase, a, b});
        }
    }
};

void prof_collect(tlsq_handle* h) {      // call after the stream was synchronised
    if (!h->prof) return;
    for (auto& sp : h->spans) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) {
            h->phase_ms[sp.phase] += ms;
            h->phase_calls[sp.phase] += 1;
        }
    }
    h->spans.clear();
    h->ev_used = 0;
}

int allreduce(tlsq_handle* h, double* buf, size_t count, int op) {
    if (h->nranks <= 1) return TLSQ_OK;
    Phase ph(h, TLSQ_PHASE_ALLREDUCE);
    int r = g_nccl.allreduce(buf, buf, count, kNcclFloat64, op, h->comm, h->stream);
    if (r != 0) return set_err(TLSQ_ERR_NCCL, "ncclAllReduce failed: %s", g_nccl.errstr ? g_nccl.errstr(r) : "?");
    return TLSQ_OK;
}

int use_device(tlsq_handle* h) {
    if (!h) return set_err(TLSQ_ERR_ARG, "null handle");
    CK(cudaSetDevice(h->device));
    t_pool = h->pool;
    return TLSQ_OK;
}

// ----------------------------------------------------------------------------------------------------------
// Host-only planning logic, shared by the solver and by the CPU test-suite (tlsq_plan_* in the C ABI).
// ----------------------------------------------------------------------------------------------------------
// votes_sum = sum over the ranks of {can_legacy, can_fused, wants_fused, wants_inplace} (0/1 each).  The per-iteration
// pipelines issue different collectives, so every rank must derive the SAME choice from the summed votes.
struct PipelineChoice { bool fused, use_w, all_legacy, all_fused, inplace_vote; };
PipelineChoice choose_pipeline(int nranks, const double* votes_sum, int env_fused /* -1: unset */) {
    PipelineChoice c;
    c.all_legacy = votes_sum[0] > (double)nranks - 0.5;
    c.all_fused = votes_sum[1] > (double)nranks - 0.5;
    if (env_fused >= 0) c.fused = c.all_fused && env_fused != 0;
    else c.fused = c.all_fused && (votes_sum[2] > 0.5 || !c.all_legacy);
    c.use_w = c.all_legacy && !c.fused;            // neither: generic kernels on every rank
    c.inplace_vote = votes_sum[3] > 0.5;           // any rank short of memory -> all ranks update Y in place
    return c;
}

// Row shards of the K Hankel rows of lowrankfilter: multiples of 32 rows (TMA / tile friendly), the last rank takes
// the remainder; tiny problems fall back to a plain split.
void shard_hankel_rows(int64_t K, int nranks, int rank, int64_t* r0, int64_t* Kl) {
    int64_t per = ((K + nranks - 1) / nranks + 31) / 32 * 32;
    if (per * (nranks - 1) >= K) per = K / nranks;
    *r0 = per * rank;
    *Kl = (rank == nranks - 1) ? K - *r0 : per;
}

struct RpcaParams {
    double lambda, tol, rho;
    int64_t maxrank, iters;
    uint32_t flags;
};
struct RpcaOut {
    double* A = nullptr;  double* E = nullptr;  double* U = nullptr;  double* S = nullptr;  double* Vt = nullptr;
    int64_t* sv = nullptr;  int64_t* iters_done = nullptr;  int32_t* converged = nullptr;  double* hist = nullptr;
    // lowrankfilter: anti-diagonal sums of the final (factored) A over this shard's Hankel rows [uh_r0, uh_r0 + M)
    double* uh_sum = nullptr;  int64_t uh_r0 = 0;  int64_t uh_Ns = 0;
    // host-buffer entry points: pinned or pageable HOST destinations of A / E.  When set, their device->host copies are
    // issued on the side stream as soon as the output pass has produced them, i.e. they overlap the eigensolver and the
    // SVD refinement that still run on the main stream; *host_copied tells the caller that they were taken care of.
    double* hA = nullptr;  double* hE = nullptr;  bool* host_copied = nullptr;
};

int gram_dense(tlsq_handle* h, const double* X, int64_t M, int64_t n, double* G);

// ----------------------------------------------------------------------------------------------------------
// rpca core: M (local rows) x N, M_global >= N, N <= kEigMaxN.  D may be dense or an implicit Hankel signal.
// All outputs are DEVICE pointers (nullable) except sv / iters_done / converged / hist (host).
// ----------------------------------------------------------------------------------------------------------
constexpr int kRetryTwoPhase = -7701;      // internal: rerun with the two-phase iteration forced from *escape_at on

int rpca_core_once(tlsq_handle* h, MatSrc D, bool hankel, int64_t M, int64_t N, const RpcaParams& p, const RpcaOut& o,
                   int64_t two_phase_from, int64_t* escape_at) {
    cudaStream_t st = h->stream;
    const int sms = h->sm_count;
    int64_t* L = &h->launches;
    const int n = (int)N;
    const size_t mn = (size_t)M * (size_t)N;
    const int nonnegA = (p.flags & TLSQ_NONNEG_A) ? 1 : 0;
    const int nonnegE = (p.flags & TLSQ_NONNEG_E) ? 1 : 0;
    const int nukeA = (p.flags & TLSQ_NO_NUKE_A) ? 0 : 1;
    const bool exact_cost = (p.flags & TLSQ_EXACT_COST) != 0;
    // hankel=true (:214-216, 234-236): anti-diagonal soft threshold of the iterate -- dense iterate, generic kernels
    const bool hk = (p.flags & TLSQ_HANKEL) != 0;
    if (hk && h->nranks > 1)
        return set_err(TLSQ_ERR_UNSUPPORTED, "rpca: hankel=true is not available on row-sharded problems");

    // global row count (for the Frobenius bracket: d = min(M_global, N))
    double Mg = (double)M;
    GramPlan plan = gram_plan(M, N, sms);
    // Three per-iteration pipelines, fastest first:
    //   fused  (n = 256)  ONE kernel per iteration: epilogue of iteration k + Gram of the SVT input of iteration k+1
    //                     (fused.cu); W is never materialised, the iterate is factored, 3 S of HBM traffic;
    //   use_w             streaming epilogue that materialises W_{k+1} + TMA-fed DMMA SYRK of W (stream.cu, syrk_tma.cu);
    //   generic           tile epilogue + Gram formed on the fly (epilogue.cu, gram.cu) for small / odd shapes.
    const bool syrk_ok = syrk_tma_eligible(reinterpret_cast<const double*>(uintptr_t(256)), M, N, M);
    SyrkPlan splan = syrk_plan(M, N, sms);
    const size_t part_bytes = syrk_ok && splan.partial_bytes > plan.partial_bytes ? splan.partial_bytes
                                                                                  : plan.partial_bytes;
    // Factored iterate: the low-rank iterate is kept as A_k = clamp(T_k V_k') (T: M x 32, V: N x 32).  The dense A is
    // then neither read nor written inside the loop; it is materialised only for the outputs, or for good (one-way
    // switch to the dense representation) if the rank estimate ever exceeds 32.
    // Pipeline choice: the one-pass kernel needs S (Y in place) .. 2 S of device memory, the two-kernel pipeline up to
    // 4 S (Y x 2, W, Z); on B200 the two-kernel pipeline is currently the faster one when it fits (profiles/), so the
    // one-pass kernel is taken when memory asks for it, when the two-kernel pipeline is not available (odd row count
    // of an implicit Hankel shard) or when TLSQ_FUSED=1 forces it.  The choice MUST be the same on every rank of a
    // sharded solve (the pipelines issue different collectives), so the local capabilities and wishes are summed over
    // the ranks first.
    auto device_free_bytes = [&]() -> size_t {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return 0; }
        cudaMemPool_t pool = h->pool;
        if (pool || cudaDeviceGetDefaultMemPool(&pool, h->device) == cudaSuccess) {
            uint64_t reserved = 0, used = 0;
            cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved);
            cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used);
            if (reserved > used) free_b += (size_t)(reserved - used);
        }
        return free_b;
    };
    const size_t free_b = device_free_bytes();
    const size_t ws_bytes = (size_t)4 << 30;
    bool can_fused = !hk && fused_eligible(D, hankel, M, N);
    if (can_fused && !syrk_ok && (o.A || o.E || o.U || o.S || o.Vt)) can_fused = false;   // padded leading dimension: factored outputs only
    // large embeddings (n > 512): always the two-kernel pipeline on a materialised W (column-chunked streaming epilogue,
    // T = W V_r by GEMM); the Gram takes the TMA SYRK when the shape allows it, else the generic DMMA kernel on W
    const bool large_n = N > kEigSmallN;
    if (large_n && hk) t_dense_fallback = true;           // host-buffer solves repeat on the dense device path
    if (large_n && hk)
        return set_err(TLSQ_ERR_UNSUPPORTED, "rpca: hankel=true is limited to min(M,N) <= %d", kEigSmallN);
    const bool can_legacy = (syrk_ok || large_n) && !hk;
    const bool wants_fused = 4 * mn * 8 + mn * 2 + ws_bytes > free_b;      // Y x 2, W, Z (+ factors) do not fit
    const bool wants_inplace = 2 * mn * 8 + mn * 2 + ws_bytes > free_b;    // not even two copies of Y fit
    double votes[5] = {(double)M, can_legacy ? 1.0 : 0.0, can_fused ? 1.0 : 0.0, wants_fused ? 1.0 : 0.0,
                       wants_inplace ? 1.0 : 0.0};
    if (h->nranks > 1) {
        DevBuf bVote;
        CK(bVote.alloc(8 * 8, st));
        for (int i = 0; i < 5; ++i) h->h_pin[i] = votes[i];
        CK(cudaMemcpyAsync(bVote.p, h->h_pin, 5 * 8, cudaMemcpyHostToDevice, st));
        CKR(allreduce(h, bVote.as<double>(), 5, kNcclSum));
        CK(cudaMemcpyAsync(h->h_pin, bVote.p, 5 * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (int i = 0; i < 5; ++i) votes[i] = h->h_pin[i];
    }
    Mg = votes[0];
    const char* env_f = getenv("TLSQ_FUSED");
    const PipelineChoice pc = choose_pipeline(h->nranks, votes + 1, env_f ? (atoi(env_f) != 0 ? 1 : 0) : -1);
    const bool all_legacy = pc.all_legacy;
    bool fused = pc.fused;
    bool use_w = pc.use_w;
    // the one-pass kernel moves Y / T tiles with TMA (16-byte strides): an odd row count gets a padded leading dimension
    const int64_t ldp = fused ? M + (M & 1) : M;
    bool fact = use_w || fused;
    DevBuf bMean;
    double* meanbuf = nullptr;
    if (hk) { CK(bMean.alloc((size_t)(M + N) * 8, st)); meanbuf = bMean.as<double>(); }
    DevBuf bW, bT0, bT1, bV0, bV1, bFp;
    double* Wbuf = nullptr;
    auto ensure_w = [&]() -> cudaError_t {
        if (Wbuf) return cudaSuccess;
        cudaError_t e = bW.alloc(mn * 8, st);
        Wbuf = bW.as<double>();
        return e;
    };
    if (use_w) CK(ensure_w());
    double* Tb[2] = {nullptr, nullptr};
    double* Vb[2] = {nullptr, nullptr};
    int svpb[2] = {0, 0};
    if (fact) {
        CK(bT0.alloc((size_t)ldp * kStreamMaxRank * 8, st)); CK(bT1.alloc((size_t)ldp * kStreamMaxRank * 8, st));
        CK(bV0.alloc((size_t)N * kStreamMaxRank * 8, st)); CK(bV1.alloc((size_t)N * kStreamMaxRank * 8, st));
        Tb[0] = bT0.as<double>(); Tb[1] = bT1.as<double>(); Vb[0] = bV0.as<double>(); Vb[1] = bV1.as<double>();
        CK(cudaMemsetAsync(Tb[0], 0, (size_t)ldp * kStreamMaxRank * 8, st));
        CK(cudaMemsetAsync(Tb[1], 0, (size_t)ldp * kStreamMaxRank * 8, st));
    }
    FusedArgs fa = {};
    if (fused) {
        CK(bFp.alloc(fused_partial_doubles(sms) * 8, st));
        fa.D = D; fa.M = M; fa.ldy = ldp; fa.ldt = ldp; fa.nonnegA = nonnegA; fa.nonnegE = nonnegE;
        fa.partial = bFp.as<double>();
        fa.zpart = fa.partial + (size_t)(sms / 2) * n * n;
    }

    DevBuf bA0, bA1, bY0, bY1, bPart, bG, bGn, bG2, bVs, bVs2, bLam, bLam2, bSig, bF, bEig, bScal, bSvp;
    // dense A ping-pong (reusing the caller's A buffer as one side when given); allocated lazily in factored mode
    double* Abuf[2] = {nullptr, nullptr};
    auto alloc_dense_a = [&]() -> cudaError_t {
        cudaError_t e = cudaSuccess;
        if (!Abuf[0]) {
            if (o.A) Abuf[0] = o.A;
            else { e = bA0.alloc(mn * 8, st); Abuf[0] = bA0.as<double>(); }
        }
        if (e == cudaSuccess && !Abuf[1]) { e = bA1.alloc(mn * 8, st); Abuf[1] = bA1.as<double>(); }
        return e;
    };
    if (!fact) CK(alloc_dense_a());
    // Dual variable: two buffers (Y_{k-1} stays available for E_k, U and the exact stop test) unless the caller needs
    // none of those outputs and two copies do not fit (lowrankfilter on very long signals): then Y is updated in place.
    bool inplace_y = false;
    if (fused && !o.E && !o.U && !o.S && !o.Vt) {
        const char* env_ip = getenv("TLSQ_INPLACE_Y");      // test hook
        inplace_y = env_ip ? atoi(env_ip) != 0 : pc.inplace_vote;     // (any rank short of memory -> all in place)
    }
    CK(bY0.alloc((size_t)ldp * N * 8, st));
    if (!inplace_y) CK(bY1.alloc((size_t)ldp * N * 8, st));
    double* Ybuf[2] = {bY0.as<double>(), inplace_y ? bY0.as<double>() : bY1.as<double>()};
    CK(bPart.alloc(part_bytes, st));
    // Gram of a materialised M x N matrix (W, Z): TMA-fed SYRK, or the generic DMMA kernel when the shape is not
    // TMA-eligible (odd leading dimension, few rows)
    auto gram_mat = [&](const double* X, double* Gdst) -> int {
        if (syrk_ok) {
            CK(launch_syrk_tma(X, M, N, M, splan, bPart.as<double>(), Gdst, st, L));
        } else {
            GramSrc g2;
            g2.D = MatSrc{X, M}; g2.A = nullptr; g2.Y = nullptr; g2.A2 = nullptr; g2.ldw = M; g2.M = M; g2.N = N;
            g2.im = 0.0; g2.eps = 0.0; g2.nonnegE = 0;
            CK(launch_gram(g2, GRAM_D, false, plan, bPart.as<double>(), Gdst, st, L));
        }
        return TLSQ_OK;
    };
    // N x 32 scratch of the column-chunked streaming epilogue (V_r diag(f) as a GEMM operand): needed whenever two
    // N x RP blocks of V do not fit in shared memory, which starts at N = 512 with a rank estimate above 24
    DevBuf bVf;
    CK(bVf.alloc((size_t)N * kStreamMaxRank * 8, st));
    CK(bG.alloc(((size_t)n * n + 8) * 8, st)); CK(bGn.alloc(((size_t)n * n + 8) * 8, st));
    CK(bG2.alloc(((size_t)n * n + 8) * 8, st));
    CK(bVs.alloc((size_t)n * n * 8, st)); CK(bVs2.alloc((size_t)n * n * 8, st));
    CK(bLam.alloc((size_t)n * 8, st)); CK(bLam2.alloc((size_t)n * 8, st));
    CK(bSig.alloc((size_t)n * 8, st)); CK(bF.alloc((size_t)n * 8, st));
    CK(bEig.alloc(eig_work_doubles(n) * 8, st));
    CK(bScal.alloc(16 * 8, st)); CK(bSvp.alloc(16, st));
    // Gram ping-pong: Gb[gi] holds the Gram of the current iteration's SVT input while the next one (one-pass kernel,
    // run-ahead) is formed in the other buffer -- so the last iteration's Gram survives for the returned SVD (:238).
    // Slot [n*n] carries ||Z||_F^2 in the packed all-reduce of the one-pass pipeline.
    double* Gb[2] = {bG.as<double>(), bGn.as<double>()};
    int gi = 0;
    double* G2 = bG2.as<double>();
    double* Vs = bVs.as<double>(); double* Vs2 = bVs2.as<double>();
    double* lam = bLam.as<double>(); double* lam2 = bLam2.as<double>();
    double* sigma = bSig.as<double>(); double* fvec = bF.as<double>();
    double* dscal = bScal.as<double>(); int* dsvp = bSvp.as<int>();
    EigWork ew;
    {
        double* base = bEig.as<double>();
        const size_t np = (size_t)n + 34;
        ew.X0 = base; base += (size_t)n * n;
        ew.Xo = base; base += np * n;
        ew.Vo = base; base += np * n;
        ew.lam_raw = base; base += np;
        ew.perm = reinterpret_cast<int*>(base); base += n;
        ew.info = reinterpret_cast<int*>(base);
    }
    double* hp = h->h_pin;
    // fast eigen path state (dominant-subspace iteration, see eig_fast.cu)
    const bool fast_ok = eig_fast_supported(n);
    DevBuf bFast;
    EigFastWork fw = {};
    if (fast_ok) {
        CK(bFast.alloc(eig_fast_work_doubles(n) * 8, st));
        fw = eig_fast_carve(bFast.as<double>(), n);
    }
    bool have_q = false;
    bool last_was_fast = false;
    int cur_bw = large_n ? 32 : 16;     // large embeddings always iterate on the 32-column block (eig_fast.cu)
    int si_budget = 12;           // subspace steps launched per iteration: last iteration's count + margin
    // exact stop test: Z is materialised by the epilogue when the Frobenius bracket is expected to be undecided, its
    // Gram runs on the TMA SYRK kernel and lambda_max is bracketed by repeated squaring
    DevBuf bZ, bSq;
    double* Zbuf = nullptr;
    CK(bSq.alloc(((size_t)2 * n * n + 32) * 8, st));
    double* sqA = bSq.as<double>();
    double* sqB = sqA + (size_t)n * n;
    double* sqf = sqB + (size_t)n * n;         // 16 f2 + 2 bounds
    double prev_fro = 1.0e300, prev_prev_fro = 1.0e300;

    // ---- setup (:174-185) --------------------------------------------------------------------------------
    CK(cudaMemsetAsync(dscal, 0, 16 * 8, st));
    if (Mg < (double)N) return set_err(TLSQ_ERR_UNSUPPORTED, "internal: rpca_core needs M >= N");
    const double dmin = (double)N;

    GramSrc gs;
    gs.D = D; gs.A = nullptr; gs.Y = nullptr; gs.A2 = nullptr; gs.ldw = M; gs.M = M; gs.N = N;
    gs.im = 0.0; gs.eps = 0.0; gs.nonnegE = nonnegE;
    {
        Phase ph(h, TLSQ_PHASE_INIT);
        if (syrk_ok && !hankel && syrk_tma_eligible(D.p, M, N, D.ld)) {
            CK(launch_syrk_tma(D.p, M, N, D.ld, splan, bPart.as<double>(), Gb[0], st, L));   // D'D
        } else if (fused) {
            FusedArgs f0 = fa;
            f0.gram_of = FUSED_GRAM_D;
            CK(launch_alm_fused(f0, hankel, nullptr, nullptr, nullptr, Gb[0], nullptr, sms, st, L));
        } else {
            CK(launch_gram(gs, GRAM_D, hankel, plan, bPart.as<double>(), Gb[0], st, L));
        }
        CKR(allreduce(h, Gb[0], (size_t)n * n, kNcclSum));
        CK(launch_maxabs(D, hankel, M, N, dscal + 1, sms, st, L));                       // norm(Y, Inf)   :178
        CKR(allreduce(h, dscal + 1, 1, kNcclMax));
        // opnorm(Y) (:177) needs only lambda_max(D'D): dominant-subspace iteration from a cold start with a
        // certificate that theta_1 is the largest eigenvalue; the full Jacobi is the fallback
        if (fast_ok) {
            CK(launch_init_block(fw.Qb, n, st, L));
            CK(launch_eig_fast(Gb[0], n, 0.0, 1, fw, lam, Vs, sigma, fvec, dsvp, st, L, 1, cur_bw));
            CK(launch_eigh(Gb[0], n, nullptr, ew, lam, Vs, sms, st, L, fw.flags));
            CK(launch_copy_block(Vs, n, fw.Qb, fw.flags, st, L));
            have_q = true;
        } else {
            CK(launch_eigh(Gb[0], n, nullptr, ew, lam, Vs, sms, st, L));
        }
    }
    CK(cudaMemcpyAsync(hp, lam, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(hp + 1, dscal + 1, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const double norm2 = sqrt(hp[0] > 0.0 ? hp[0] : 0.0);
    const double norminf = hp[1] / p.lambda;
    const double dual_norm = norm2 > norminf ? norm2 : norminf;                          // :179
    const double d_norm = norm2;                                                         // :180
    double mu = 1.25 / norm2;                                                            // :182
    const double mubar = mu * 1.0e7;                                                     // :183
    bool gram_ready = false;       // G already holds the Gram of this iteration's SVT input (fused path)
    {
        Phase ph(h, TLSQ_PHASE_INIT);
        CK(launch_init_ya(D, hankel, M, N, dual_norm, Ybuf[0], fact ? nullptr : Abuf[0], fused ? nullptr : Wbuf,
                          1.0 / mu, p.lambda / mu, nonnegE, sms, st, L, ldp));           // Y ./= dual_norm :181
        if (fused) {
            // Gram of the first SVT input W_1 = (D - E_1) + Y_0/mu_1 (A_0 = 0), formed on the fly
            FusedArgs f1 = fa;
            f1.gram_of = FUSED_GRAM_W; f1.im = 1.0 / mu; f1.eps = p.lambda / mu;
            CK(launch_alm_fused(f1, hankel, Ybuf[0], nullptr, nullptr, Gb[0], nullptr, sms, st, L));
            CKR(allreduce(h, Gb[0], (size_t)n * n, kNcclSum));
            gram_ready = true;
        }
    }

    int cur = 0;
    int64_t k_done = 0;
    int conv = 0;
    int svp_last = 10;
    double im_last = 0.0, eps_last = 0.0;
    int prev_idx = 0, last_idx = 0;
    static const bool dbg_eig = getenv("TLSQ_DEBUG_EIG") != nullptr;
    // Host/device overlap of the two-kernel pipeline (no blocking host sync between the eigen step and the epilogue, and
    // none between the epilogue and the next Gram):
    //  * the streaming epilogue is launched on a GUESS of the rank (the previous iteration's) and reads the actual svp
    //    from device memory; a guess that turns out too small makes the kernels return untouched and is relaunched;
    //  * while the host waits for ||Z||_F^2 of iteration k, the Gram and the eigen step of iteration k+1 are already
    //    enqueued ("run-ahead"; skipped when iteration k may converge, so at most nothing is wasted in practice).
    const bool no_ahead = getenv("TLSQ_NO_RUNAHEAD") != nullptr;
    const bool trace = getenv("TLSQ_TRACE") != nullptr;
    auto now_us = []() {
        struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
        return (double)ts.tv_sec * 1e6 + (double)ts.tv_nsec * 1e-3;
    };
    double t_iter0 = now_us();
    int svp_pred = 0;              // rank guess for the coming iteration (from the leading eigenvalues of the last one)
    bool ahead_done = false;       // Gram + eigen step of the coming iteration are already enqueued
    bool eig_stale = false;        // lam / Vs / sigma belong to a run-ahead eigen step, not to the last finished iteration
    int64_t n_redo = 0;

    // eigen step of one iteration on Gsrc: sigma, V_r, svp = #{sigma >= im}  (:193-204)
    auto enqueue_eig = [&](const double* Gsrc, double im_k) -> int {
        Phase ph(h, TLSQ_PHASE_EIG);
        // a 16-column block is enough while the rank estimate stays <= 10 (it must stay <= block - 2); widening
        // the block needs an orthonormal 32-column basis, which the next full Jacobi provides
        const int want_bw = svp_last <= 10 ? 16 : 32;
        if (want_bw > cur_bw) { have_q = false; cur_bw = 32; }
        const bool block_fits = cur_bw <= eig_fast_max_block(n);      // n > 256: only the 16-column block
        if (fast_ok && have_q && block_fits) {
            // dominant eigenpairs + certified count; the full Jacobi below only runs (device-side flag) when the
            // fast path could not prove the count
            CK(launch_eig_fast(Gsrc, n, im_k, nukeA, fw, lam, Vs, sigma, fvec, dsvp, st, L, 0, cur_bw, si_budget));
            CK(launch_eigh(Gsrc, n, nullptr, ew, lam, Vs, sms, st, L, fw.flags));
            CK(launch_svt_post(lam, n, im_k, nukeA, sigma, fvec, dsvp, st, L, fw.flags));   // :198
            CK(launch_copy_block(Vs, n, fw.Qb, fw.flags, st, L));
            last_was_fast = true;
        } else {
            CK(launch_eigh(Gsrc, n, nullptr, ew, lam, Vs, sms, st, L));
            CK(launch_svt_post(lam, n, im_k, nukeA, sigma, fvec, dsvp, st, L));          // :198
            if (fast_ok) { CK(launch_copy_block(Vs, n, fw.Qb, nullptr, st, L)); have_q = true; }
            last_was_fast = false;
        }
        return TLSQ_OK;
    };

    for (int64_t k = 1; k <= p.iters; ++k) {                                             // :186
        const int nxt = cur ^ 1;
        const double im = 1.0 / mu;
        const double eps = p.lambda / mu;
        double* G = Gb[gi];
        double* Gnext = Gb[gi ^ 1];
        // SVT input Gram  (:188-194)
        gs.A = Abuf[cur]; gs.Y = Ybuf[cur]; gs.A2 = nullptr; gs.im = im; gs.eps = eps;
        if (!ahead_done) {
            if (!gram_ready) {
                {
                    Phase ph(h, TLSQ_PHASE_GRAM);
                    if (use_w) CKR(gram_mat(Wbuf, G));
                    else CK(launch_gram(gs, GRAM_W, hankel, plan, bPart.as<double>(), G, st, L));
                }
                CKR(allreduce(h, G, (size_t)n * n, kNcclSum));
            }
            CKR(enqueue_eig(G, im));
        }
        gram_ready = false;
        ahead_done = false;
        eig_stale = false;
        bool was_fast_k = last_was_fast;
        const double mu_next = fmin(mu * p.rho, mubar);                                  // :223
        int svp = 0;
        // The streaming / fused kernels are specialised on the rank.  Two-kernel pipeline: launch on a guess (the last
        // rank seen) and let the kernels check it; first iteration and the one-pass pipeline: fetch svp (short host sync).
        bool svp_known = false;
        int svp_guess = svp_pred > svp_last ? svp_pred : svp_last;
        const bool speculate = use_w && k > 1;
        if ((use_w || fused) && !speculate) {
            CK(cudaMemcpyAsync(hp + 1, dsvp, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            memcpy(&svp, hp + 1, 4);
            svp_known = true;
            svp_guess = svp;
        }
        // will the Frobenius bracket [fro/sqrt(d), fro] probably straddle tol?  (fro shrinks by < 8x per iteration)
        bool want_z = (use_w || fused) && (exact_cost || (p.tol > 0.0 && prev_fro < 8.0 * sqrt(dmin) * p.tol));
        if (fused) {
            // One-pass pipeline.  With two Y buffers nothing is predicted: the normal pass runs, and only when the
            // Frobenius bracket cannot decide is Z'Z formed after the fact from (Y_{k-1}, T_{k-1}, T_k).  With Y in
            // place Y_{k-1} is gone after the pass, so iterations that may need ||Z||_2 run in two phases; the
            // prediction extrapolates the last observed decay (4x safety) instead of assuming a fixed 8x.
            if (!inplace_y) want_z = false;
            else if (!exact_cost && p.tol > 0.0 && prev_prev_fro < 1.0e299) {
                const double ratio = fmin(prev_fro / prev_prev_fro, 1.0);
                want_z = prev_fro * ratio < 4.0 * sqrt(dmin) * p.tol;
            }
            const bool no_pred = getenv("TLSQ_NO_PREDICT_Z") != nullptr;     // test hook: exercise the retry below
            if (inplace_y && no_pred && !exact_cost) want_z = false;
            if (inplace_y && k >= two_phase_from) want_z = true;
        }
        if (fused && (svp > kFusedMaxRank || svpb[cur] > kFusedMaxRank)) {
            // rank estimate beyond the fused kernel: materialise W_k once and continue on the streaming pipeline
            if (ldp != M || inplace_y || !all_legacy)
                return set_err(TLSQ_ERR_UNSUPPORTED, "rpca: rank estimate %d exceeds the one-pass kernel's %d and the "
                               "streaming pipeline cannot take over (padded / in-place dual variable)", svp, kFusedMaxRank);
            CK(ensure_w());
            EpiArgs wa = {};
            wa.D = D; wa.Yp = Ybuf[cur]; wa.Tp = Tb[cur]; wa.Vp = Vb[cur]; wa.svp_prev = svpb[cur];
            wa.Tn = Tb[cur]; wa.Vs = Vb[cur]; wa.M = M; wa.N = N; wa.ldw = M; wa.im = im; wa.eps = eps;
            wa.nonnegA = nonnegA; wa.nonnegE = nonnegE;
            CK(launch_final_from_factors(wa, hankel, svpb[cur], Wbuf, sms, st, L));
            fused = false;
            use_w = true;
        }

        double zz = 0.0;
        bool z_gram_ready = false;     // G2 holds Z_k'Z_k (fused path, two-phase iteration)
        bool y_written = true;
        EpiArgs ea = {};
        if (fused) {
            // ---- one-pass iteration (fused.cu) ----------------------------------------------------------------------
            FusedArgs f = fa;
            f.Vp = Vb[cur]; f.svp_prev = svpb[cur]; f.Vs = Vs; f.fvec = fvec; f.svp = svp;
            f.Yn = Ybuf[nxt]; f.Tn = Tb[nxt];
            f.im = im; f.eps = eps; f.mu = mu; f.im_next = 1.0 / mu_next; f.eps_next = p.lambda / mu_next;
            if (want_z) {
                // phase A of an iteration whose stop test probably needs opnorm(Z): T_k, ||Z||_F^2 and Z'Z; Y is not
                // touched yet, so that (Y_{k-1}, T_{k-1}, T_k) still describe the solution if this iteration converges
                Phase ph(h, TLSQ_PHASE_EXACT_COST);
                f.gram_of = FUSED_GRAM_Z; f.compute_T = 1; f.write_Y = 0;
                CK(launch_alm_fused(f, hankel, Ybuf[cur], Tb[cur], nullptr, G2, G2 + (size_t)n * n, sms, st, L));
                CKR(allreduce(h, G2, (size_t)n * n + 1, kNcclSum));
                CK(cudaMemcpyAsync(hp, G2 + (size_t)n * n, 8, cudaMemcpyDeviceToHost, st));
                z_gram_ready = true;
                y_written = false;
            } else {
                Phase ph(h, TLSQ_PHASE_FUSED);
                f.gram_of = FUSED_GRAM_WNEXT; f.compute_T = 1; f.write_Y = 1;
                CK(launch_alm_fused(f, hankel, Ybuf[cur], Tb[cur], nullptr, Gnext, Gnext + (size_t)n * n, sms, st, L));
                CKR(allreduce(h, Gnext, (size_t)n * n + 1, kNcclSum));
                CK(cudaMemcpyAsync(hp, Gnext + (size_t)n * n, 8, cudaMemcpyDeviceToHost, st));
                gram_ready = true;
            }
            CK(cudaMemcpyAsync(Vb[nxt], Vs, (size_t)N * kStreamMaxRank * 8, cudaMemcpyDeviceToDevice, st));
            svpb[nxt] = svp;
            CK(cudaMemcpyAsync(hp + 1, dsvp, 4, cudaMemcpyDeviceToHost, st));
            if (dbg_eig) {
                CK(cudaMemcpyAsync(hp + 2, ew.info, 4, cudaMemcpyDeviceToHost, st));
                if (fast_ok) CK(cudaMemcpyAsync(hp + 4, fw.flags, 32, cudaMemcpyDeviceToHost, st));
            }
            if (fast_ok && was_fast_k) CK(cudaMemcpyAsync(hp + 8, fw.flags, 16, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
        } else {
            // ---- epilogue of the two-kernel pipelines  (:188-192, 205-222) -----------------------------------------
            for (int attempt = 0;; ++attempt) {
                CK(cudaMemsetAsync(dscal, 0, 8, st));
                ea = EpiArgs{};
                ea.D = D; ea.Ap = Abuf[cur]; ea.Yp = Ybuf[cur]; ea.An = Abuf[nxt]; ea.Yn = Ybuf[nxt];
                ea.Eout = nullptr; ea.Uout = nullptr; ea.M = M; ea.N = N; ea.ldw = M; ea.Vs = Vs; ea.fvec = fvec;
                ea.svp = dsvp; ea.im = im; ea.eps = eps; ea.mu = mu; ea.nonnegA = nonnegA; ea.nonnegE = nonnegE;
                ea.zz = dscal;
                if (want_z && !Zbuf && !inplace_y) { CK(bZ.alloc(mn * 8, st)); Zbuf = bZ.as<double>(); }
                ea.Zout = (want_z && Zbuf) ? Zbuf : nullptr;
                ea.Wn = Wbuf; ea.im_next = 1.0 / mu_next; ea.eps_next = p.lambda / mu_next;
                ea.vf_work = bVf.as<double>();
                if (large_n && svp_guess > kStreamMaxRank) t_dense_fallback = true;
                if (large_n && svp_guess > kStreamMaxRank)
                    return set_err(TLSQ_ERR_UNSUPPORTED, "rpca: rank estimate %d > %d with min(M,N) = %lld > %d is outside "
                                   "the accelerated path", svp_guess, kStreamMaxRank, (long long)N, kEigSmallN);
                bool guarded = false;          // the launch below checks the rank guess on the device
                int rp_launched = 0;
                {
                    Phase ph(h, TLSQ_PHASE_EPILOGUE);
                    if (fact && !stream_factored_fits(N, svp_guess, svpb[cur])) {
                        // rank estimate beyond the factored kernels: materialise A_{k-1} and continue with the dense iterate
                        CK(alloc_dense_a());
                        CK(launch_fact_to_dense(Tb[cur], Vb[cur], svpb[cur], M, N, nonnegA, Abuf[cur], sms, st, L));
                        ea.Ap = Abuf[cur]; ea.An = Abuf[nxt];
                        fact = false;
                    }
                    if (fact) {
                        ea.Tp = Tb[cur]; ea.Vp = Vb[cur]; ea.svp_prev = svpb[cur]; ea.Tn = Tb[nxt];
                        CK(launch_stream_epilogue(ea, Wbuf, svp_guess, hankel, sms, st, L, !svp_known));
                        guarded = !svp_known;
                        rp_launched = stream_rank_pad(svp_guess, svpb[cur], true);
                        // V_k of this iterate (Vs is overwritten by the next eigen-decomposition)
                        CK(cudaMemcpyAsync(Vb[nxt], Vs, (size_t)N * kStreamMaxRank * 8, cudaMemcpyDeviceToDevice, st));
                    } else if (use_w && svp_guess <= kStreamMaxRank) {
                        CK(launch_stream_epilogue(ea, Wbuf, svp_guess, hankel, sms, st, L, !svp_known));
                        guarded = !svp_known;
                        rp_launched = stream_rank_pad(svp_guess, 0, false);
                    } else if (hk) {
                        // A_raw = U_r (S_r - 1/mu) V_r' ; soft_hankel!(A, lambda/mu) ; clamp ; Z ; Y   (:205-222)
                        ea.raw_only = 1;
                        CK(launch_epilogue(ea, hankel, false, sms, st, L));
                        CK(launch_unhankel(ea.An, M, N, 1, M + N - 1, meanbuf, st, L));          // anti-diagonal means
                        CK(launch_hankel_finish(ea, hankel, meanbuf, sms, st, L));
                    } else {
                        CK(launch_epilogue(ea, hankel, false, sms, st, L));
                    }
                }
                CKR(allreduce(h, dscal, 1, kNcclSum));
                CK(cudaMemcpyAsync(hp, dscal, 8, cudaMemcpyDeviceToHost, st));
                CK(cudaMemcpyAsync(hp + 1, dsvp, 4, cudaMemcpyDeviceToHost, st));
                if (dbg_eig) {
                    CK(cudaMemcpyAsync(hp + 2, ew.info, 4, cudaMemcpyDeviceToHost, st));
                    if (fast_ok) CK(cudaMemcpyAsync(hp + 4, fw.flags, 32, cudaMemcpyDeviceToHost, st));
                }
                if (fast_ok && was_fast_k) CK(cudaMemcpyAsync(hp + 8, fw.flags, 16, cudaMemcpyDeviceToHost, st));
                // run-ahead: Gram + eigen step of iteration k+1 behind the epilogue, before the host looks at the result
                const bool run_ahead = use_w && !no_ahead && !want_z && k < p.iters && attempt == 0;
                const double t_enq = now_us();
                double t_ra = t_enq;
                if (run_ahead) {
                    CK(cudaEventRecord(h->ev_iter, st));
                    {
                        Phase ph(h, TLSQ_PHASE_GRAM);
                        CKR(gram_mat(Wbuf, Gnext));
                    }
                    CKR(allreduce(h, Gnext, (size_t)n * n, kNcclSum));
                    CKR(enqueue_eig(Gnext, 1.0 / mu_next));
                    ahead_done = true;
                    eig_stale = true;
                    t_ra = now_us();
                    CK(cudaEventSynchronize(h->ev_iter));
                } else {
                    CK(cudaStreamSynchronize(st));
                }
                if (trace) {
                    const double t_done = now_us();
                    fprintf(stderr, "[tlsq-trace] k=%lld attempt=%d enqueue %.0f us, run-ahead enqueue %.0f us, wait %.0f us, ahead=%d guarded=%d rp=%d\n",
                            (long long)k, attempt, t_enq - t_iter0, t_ra - t_enq, t_done - t_ra, ahead_done ? 1 : 0, guarded ? 1 : 0,
                            rp_launched);
                    t_iter0 = t_done;
                }
                int svp_dev = 0;
                memcpy(&svp_dev, hp + 1, 4);
                if (guarded && svp_dev > rp_launched) {
                    // the guess was too small: the epilogue kernels returned without touching anything.  A run-ahead
                    // eigen step has overwritten this iteration's sigma / V_r: redo it from the intact Gram.
                    ++n_redo;
                    if (ahead_done) {
                        CKR(enqueue_eig(G, im));
                        was_fast_k = last_was_fast;
                        ahead_done = false;
                        eig_stale = false;
                    }
                    svp_guess = svp_dev;
                    svp_known = true;
                    continue;
                }
                svp = svp_dev;
                break;
            }
            if (fact) svpb[nxt] = svp;
            // (A rank guess from this iteration's leading Ritz values against the next threshold was tried: the bulk sits
            // just below 1/mu_k and is above 1/mu_{k+1}, so it over-counts every iteration and costs a slower
            // specialisation -- the last rank is the better guess; a jump costs one relaunch.)
            svp_pred = svp;
        }
        if (fast_ok && was_fast_k) {
            int fl[4];
            memcpy(fl, hp + 8, 16);
            // converged in fl[3] steps: budget that + 3 next time; a fallback resets the budget
            // (a launch that exits at once costs ~2 us, a budget that is too small costs a full Jacobi: stay generous)
            si_budget = fl[1] ? 12 : (fl[3] + 4 > 8 ? fl[3] + 4 : 8);
        }
        if (dbg_eig) {
            int sw, fl[8] = {0};
            memcpy(&sw, hp + 2, 4);
            if (fast_ok) memcpy(fl, hp + 4, 32);
            fprintf(stderr, "[tlsq] iter %lld: full-jacobi sweeps %d | fast: conv %d need_full %d svp %d si_steps %d "
                            "certified %d si_sweeps %d | redo %lld ahead %d\n", (long long)k, sw, fl[0], fl[1], fl[2], fl[3],
                    fl[4], fl[5], (long long)n_redo, ahead_done ? 1 : 0);
        }
        zz = hp[0];
        memcpy(&svp, hp + 1, 4);
        svp_last = svp;
        im_last = im; eps_last = eps; prev_idx = cur; last_idx = nxt;
        // stop test  cost = opnorm(Z)/d_norm < tol   (:225-231)
        const double fro = sqrt(zz) / d_norm;        // ||Z||_F/d_norm >= cost >= ||Z||_F/(sqrt(d) d_norm)
        double cost_rec = -fro;
        bool converged = false;
        bool need_exact = exact_cost;
        if (!need_exact) {
            if (fro < p.tol) converged = true;
            else if (fro / sqrt(dmin) >= p.tol) converged = false;
            else need_exact = true;
        }
        prev_prev_fro = prev_fro;
        prev_fro = fro;
        if (need_exact && inplace_y && !z_gram_ready) {
            // Y was updated in place and the prediction missed an undecided Frobenius bracket: Z_k cannot be rebuilt from
            // Y_k alone.  The solve is deterministic and D is never modified, so it is simply repeated with the two-phase
            // iteration forced from this iteration on -- the stopping iteration always equals the reference's (:225-231).
            *escape_at = k;
            CK(cudaStreamSynchronize(st));
            return kRetryTwoPhase;
        }
        if (need_exact) {
            Phase ph(h, TLSQ_PHASE_EXACT_COST);
            if (z_gram_ready) {
                // G2 = Z'Z came with phase A
            } else if (fused) {
                // the bracket was not predicted: Z_k'Z_k from (Y_{k-1}, T_{k-1}, T_k), nothing written
                FusedArgs f = fa;
                f.Vp = Vb[cur]; f.svp_prev = svpb[cur]; f.Vs = Vb[nxt]; f.fvec = fvec; f.svp = svp;
                f.im = im; f.eps = eps; f.mu = mu; f.gram_of = FUSED_GRAM_Z; f.compute_T = 0; f.write_Y = 0;
                CK(launch_alm_fused(f, hankel, Ybuf[cur], Tb[cur], Tb[nxt], G2, nullptr, sms, st, L));
                CKR(allreduce(h, G2, (size_t)n * n, kNcclSum));
            } else if (want_z && Zbuf) {
                CKR(gram_mat(Zbuf, G2));
                CKR(allreduce(h, G2, (size_t)n * n, kNcclSum));
            } else if (fact) {
                // the bracket was not predicted: rebuild Z_k from the factored iterates, then the same SYRK
                if (!Zbuf) { CK(bZ.alloc(mn * 8, st)); Zbuf = bZ.as<double>(); }
                ea.Vs = Vb[nxt];               // V_k (Vs may already belong to the run-ahead eigen step)
                CK(launch_z_from_factors(ea, hankel, svp, Zbuf, sms, st, L));
                CKR(gram_mat(Zbuf, G2));
                CKR(allreduce(h, G2, (size_t)n * n, kNcclSum));
            } else {
                gs.A = Abuf[cur]; gs.Y = Ybuf[cur]; gs.A2 = Abuf[nxt]; gs.im = im; gs.eps = eps;
                CK(launch_gram(gs, GRAM_Z, hankel, plan, bPart.as<double>(), G2, st, L));
                CKR(allreduce(h, G2, (size_t)n * n, kNcclSum));
            }
            // bracket lambda_max(Z'Z) by repeated squaring; only a bracket that straddles tol^2 needs the Jacobi
            CK(launch_lmax_bounds(G2, n, sqA, sqB, sqf, sqf + 16, st, L));
            CK(cudaMemcpyAsync(hp, sqf + 16, 16, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            const double c_lo = sqrt(hp[0] > 0.0 ? hp[0] : 0.0) / d_norm;
            const double c_hi = sqrt(hp[1] > 0.0 ? hp[1] : 0.0) / d_norm;
            const bool bracket_ok = (hp[0] == hp[0]) && (hp[1] == hp[1]);
            if (!exact_cost && bracket_ok && c_hi < p.tol) { converged = true; cost_rec = -c_hi; }
            else if (!exact_cost && bracket_ok && c_lo >= p.tol) { converged = false; cost_rec = -c_hi; }
            else {
                CK(launch_eigh(G2, n, nullptr, ew, lam2, Vs2, sms, st, L));
                CK(cudaMemcpyAsync(hp, lam2, 8, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
                const double cost = sqrt(hp[0] > 0.0 ? hp[0] : 0.0) / d_norm;
                cost_rec = cost;
                converged = cost < p.tol;
            }
        }
        if (o.hist) {
            o.hist[3 * (k - 1) + 0] = (double)k;
            o.hist[3 * (k - 1) + 1] = (double)svp;
            o.hist[3 * (k - 1) + 2] = cost_rec;
        }
        k_done = k;
        if (fused && !y_written && !(converged || k == p.iters)) {
            // phase B: the iteration goes on -> Y_k and the Gram of W_{k+1}, with T_k taken from phase A
            Phase ph(h, TLSQ_PHASE_FUSED);
            FusedArgs f = fa;
            f.Vp = Vb[cur]; f.svp_prev = svpb[cur]; f.Vs = Vb[nxt]; f.fvec = fvec; f.svp = svp;
            f.Yn = Ybuf[nxt]; f.Tn = nullptr;
            f.im = im; f.eps = eps; f.mu = mu; f.im_next = 1.0 / mu_next; f.eps_next = p.lambda / mu_next;
            f.gram_of = FUSED_GRAM_WNEXT; f.compute_T = 0; f.write_Y = 1;
            CK(launch_alm_fused(f, hankel, Ybuf[cur], Tb[cur], Tb[nxt], Gnext, nullptr, sms, st, L));
            CKR(allreduce(h, Gnext, (size_t)n * n, kNcclSum));
            gram_ready = true;
        }
        mu = mu_next;
        cur = nxt;
        if (converged) { conv = 1; break; }
        if (k == p.iters) break;
        if (gram_ready || ahead_done) gi ^= 1;         // the next iteration's Gram is in the other buffer
    }
    double* G = Gb[gi];                                // Gram of the LAST iteration's SVT input W_k

    // ---- outputs (:238) ----------------------------------------------------------------------------------
    Phase ph_final(h, TLSQ_PHASE_FINALIZE);
    const bool want_svd = o.S || o.Vt || o.U;
    bool d2h_pending = false;
    // The returned SVD is that of the LAST SVT input W_k (:194, 238): W_k is materialised once (the W buffer of the
    // two-kernel pipeline is free now).
    double* Wfin = nullptr;
    if (want_svd) { CK(ensure_w()); Wfin = Wbuf; }           // allocated in stream order BEFORE the fork point
    // fork point of the side stream; the eigensolver is enqueued FIRST so that its cluster kernel gets its SMs before
    // the bandwidth-bound output pass fills the machine
    CK(cudaEventRecord(h->ev_fork, st));
    if (want_svd && (eig_stale || (fast_ok && last_was_fast))) {
        // the fast path only carries the dominant block (and a run-ahead eigen step belongs to an iteration that never
        // ran); the returned SVD needs the full spectrum of W_k, whose Gram is still in G
        CK(launch_eigh(G, n, nullptr, ew, lam, Vs, sms, st, L));
        CK(launch_svt_post(lam, n, im_last, nukeA, sigma, fvec, dsvp, st, L));
    }
    if (fact) {
        // Factored iterate: ONE pass produces A_k, E_k and (for the SVD) W_k from (T_{k-1}, V_{k-1}, Y_{k-1}) and
        // (T_k, V_k).  The pass is HBM-bound and independent of the full eigen-decomposition above (latency-bound, a few
        // SMs): it runs on the side stream, concurrently.
        cudaStream_t ss = h->side;
        CK(cudaStreamWaitEvent(ss, h->ev_fork, 0));
        if (o.uh_sum)
            CK(launch_unhankel_factors(Tb[last_idx], ldp, Vb[last_idx], svpb[last_idx], nonnegA, o.uh_r0, M, N, o.uh_Ns,
                                       o.uh_sum, sms, ss, L));
        if (o.E || want_svd) {
            EpiArgs fe = {};
            fe.D = D; fe.Yp = Ybuf[prev_idx]; fe.Tp = Tb[prev_idx]; fe.Vp = Vb[prev_idx]; fe.svp_prev = svpb[prev_idx];
            fe.Tn = Tb[last_idx]; fe.Vs = Vb[last_idx]; fe.An = o.A; fe.Eout = o.E; fe.M = M; fe.N = N; fe.ldw = M;
            fe.im = im_last; fe.eps = eps_last; fe.nonnegA = nonnegA; fe.nonnegE = nonnegE;
            CK(launch_final_from_factors(fe, hankel, svpb[last_idx], Wfin, sms, ss, L));
        } else if (o.A) {
            CK(launch_fact_to_dense(Tb[last_idx], Vb[last_idx], svpb[last_idx], M, N, nonnegA, o.A, sms, ss, L));
        }
        CK(cudaEventRecord(h->ev_join, ss));
        CK(cudaStreamWaitEvent(st, h->ev_join, 0));
        if (o.host_copied && (o.hA || o.hE)) {
            if (o.hA && o.A) CK(cudaMemcpyAsync(o.hA, o.A, mn * 8, cudaMemcpyDeviceToHost, ss));
            if (o.hE && o.E) CK(cudaMemcpyAsync(o.hE, o.E, mn * 8, cudaMemcpyDeviceToHost, ss));
            CK(cudaEventRecord(h->ev_d2h, ss));
            d2h_pending = true;
        }
    } else {
        if (o.uh_sum) {
            // the rank estimate left the factored path: anti-diagonal sums from the dense A_k
            DevBuf bCnt;
            CK(bCnt.alloc((size_t)o.uh_Ns * 8, st));
            CK(cudaMemsetAsync(o.uh_sum, 0, (size_t)o.uh_Ns * 8, st));
            CK(launch_unhankel_partial(Abuf[last_idx], o.uh_r0, M, N, 1, o.uh_Ns, o.uh_sum, bCnt.as<double>(), st, L));
        }
        // NB: E and W_k are recomputed from (A_{k-1}, Y_{k-1}); A_{k-1} may live in the caller's A buffer, so they must
        // be produced before A_k is copied there.
        if (o.E || want_svd) {
            CK(launch_compute_e(D, hankel, M, N, Abuf[prev_idx], Ybuf[prev_idx], im_last, eps_last, nonnegE, o.E, sms,
                                st, L, Wfin));
            if (hk && o.E) {                                                             // soft_hankel!(E, lambda/mu) :234-236
                CK(launch_unhankel(o.E, M, N, 1, M + N - 1, meanbuf, st, L));
                CK(launch_soft_hankel_apply(o.E, M, N, meanbuf, p.lambda / mu, sms, st, L));
            }
        }
        if (o.A && Abuf[last_idx] != o.A)
            CK(cudaMemcpyAsync(o.A, Abuf[last_idx], mn * 8, cudaMemcpyDeviceToDevice, st));
    }
    if (want_svd) {
        // SVD refinement (CholeskyQR2 with the eigenvectors of the Gram as the first factor).  sigma, V from
        // eig(W'W) carry an absolute error eps*s_1^2/s_i, visible in the tail of the spectrum.  With s~ = max(s, 1e-8 s_1):
        //   C = W V diag(1/s~)            nearly orthonormal columns (DMMA GEMM)
        //   C'C = R'R                     Gram formed FROM THE DATA in the rotated, scaled basis + Cholesky
        //   K = R diag(s~) = U_K S V_K'   one-sided Jacobi of the n x n factor: K'K = V' W'W V exactly (to eps kappa(C)^2)
        //   W = (W V V_K S^-1) S (V V_K)' singular values to eps*s_1 like LAPACK's, V = V V_K, U = W V S^-1
        double* Cbuf = o.U;
        if (!Cbuf) { if (!Zbuf) { CK(bZ.alloc(mn * 8, st)); Zbuf = bZ.as<double>(); } Cbuf = Zbuf; }
        double* sc = lam2;                       // clamped scales s~
        double* Vfin = Gb[gi ^ 1];               // refined basis V V_K (free n x n scratch)
        CK(launch_scale_cols_floor(Vs, sigma, n, 1.0e-8, sqA, sc, st, L));
        CK(launch_gemm_any(Wfin, M, n, M, sqA, n, Cbuf, st, L));
        CKR(gram_dense(h, Cbuf, M, n, G2));
        CKR(allreduce(h, G2, (size_t)n * n, kNcclSum));
        CK(launch_chol_upper(G2, n, st, L));
        CK(launch_scale_cols_mul(G2, sc, n, sqB, st, L));
        CK(launch_eigh(sqB, n, nullptr, ew, sigma, Vs2, sms, st, L, nullptr, 1));
        CK(launch_gemm_nn(Vs, Vs2, n, Vfin, st, L));
        if (o.S) CK(cudaMemcpyAsync(o.S, sigma, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
        if (o.Vt) CK(launch_transpose(Vfin, N, N, o.Vt, st, L));
        if (o.U) {
            CK(launch_scale_cols_inv(Vfin, sigma, n, sqA, st, L));
            CK(launch_gemm_any(Wfin, M, n, M, sqA, n, o.U, st, L));                      // U = W_k V diag(1/s)
        }
    }
    if (d2h_pending) { CK(cudaStreamWaitEvent(st, h->ev_d2h, 0)); *o.host_copied = true; }
    CK(cudaStreamSynchronize(st));
    if (o.sv) {
        int64_t sv = svp_last;                                                           // :199-204
        if (sv < 1) sv = 1;
        if (p.maxrank > 0 && sv > p.maxrank) sv = p.maxrank;
        *o.sv = sv;
    }
    if (o.iters_done) *o.iters_done = k_done;
    if (o.converged) *o.converged = conv;
    return TLSQ_OK;
}

int rpca_core(tlsq_handle* h, MatSrc D, bool hankel, int64_t M, int64_t N, const RpcaParams& p, const RpcaOut& o) {
    int64_t two_phase_from = INT64_MAX;
    for (int attempt = 0; attempt < 4; ++attempt) {
        int64_t escape_at = 0;
        const int r = rpca_core_once(h, D, hankel, M, N, p, o, two_phase_from, &escape_at);
        if (r != kRetryTwoPhase) return r;
        two_phase_from = escape_at;
    }
    return set_err(TLSQ_ERR_CUDA, "rpca: internal error (two-phase retry did not settle)");
}

int check_rpca_args(int64_t M, int64_t N, const RpcaParams& p) {
    if (M < 1 || N < 1) return set_err(TLSQ_ERR_ARG, "rpca: empty matrix (%lld x %lld)", (long long)M, (long long)N);
    if (p.iters < 1) return set_err(TLSQ_ERR_ARG, "rpca: iters must be >= 1");
    if (!(p.lambda > 0.0)) return set_err(TLSQ_ERR_ARG, "rpca: lambda must be > 0");
    if (!(p.rho > 0.0)) return set_err(TLSQ_ERR_ARG, "rpca: rho must be > 0");
    return TLSQ_OK;
}

// dense rpca on device pointers, any orientation (M < N is solved on the transpose: the problem is
// transpose-invariant -- nuclear / l1 / spectral norms and lambda = 1/sqrt(max(M,N)) all are)
int rpca_dev(tlsq_handle* h, const double* D, int64_t M, int64_t N, const RpcaParams& p, const RpcaOut& o) {
    CKR(check_rpca_args(M, N, p));
    cudaStream_t st = h->stream;
    const bool tall = (M >= N) || h->nranks > 1;
    const int64_t nn = tall ? N : M;
    if (nn > kEigMaxN)
        return set_err(TLSQ_ERR_UNSUPPORTED, "rpca: min(M,N) = %lld exceeds the supported %d", (long long)nn,
                       kEigMaxN);
    if (tall) {
        MatSrc src{D, M};
        return rpca_core(h, src, false, M, N, p, o);
    }
    // wide: solve on D' (N x M)
    const size_t mn = (size_t)M * N;
    DevBuf bDt, bAt, bEt, bUt, bVtt;
    CK(bDt.alloc(mn * 8, st));
    CK(launch_transpose(D, M, N, bDt.as<double>(), st, &h->launches));
    RpcaOut ot = o;
    ot.A = nullptr; ot.E = nullptr; ot.U = nullptr; ot.Vt = nullptr;
    ot.hA = nullptr; ot.hE = nullptr; ot.host_copied = nullptr;       // outputs are transposed back first
    if (o.A) { CK(bAt.alloc(mn * 8, st)); ot.A = bAt.as<double>(); }
    if (o.E) { CK(bEt.alloc(mn * 8, st)); ot.E = bEt.as<double>(); }
    const int64_t d = M;                       // min(M, N)
    if (o.Vt) { CK(bUt.alloc((size_t)N * d * 8, st)); ot.U = bUt.as<double>(); }    // U' of D' is N x d  -> Vt = U''
    if (o.U) { CK(bVtt.alloc((size_t)d * d * 8, st)); ot.Vt = bVtt.as<double>(); }  // Vt' of D' is d x M -> U = Vt''
    MatSrc src{bDt.as<double>(), N};
    CKR(rpca_core(h, src, false, N, M, p, ot));
    if (o.A) CK(launch_transpose(ot.A, N, M, o.A, st, &h->launches));
    if (o.E) CK(launch_transpose(ot.E, N, M, o.E, st, &h->launches));
    if (o.Vt) CK(launch_transpose(ot.U, N, d, o.Vt, st, &h->launches));
    if (o.U) CK(launch_transpose(ot.Vt, d, M, o.U, st, &h->launches));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

int rpca_cb_host(tlsq_handle* h, const double* Dh, int64_t M, int64_t N, const RpcaParams& p, tlsq_svd_fn svd_fn,
                 tlsq_opnorm_fn opn_fn, void* user, double* Ah, double* Eh, double* Uh, double* Sh, double* Vth,
                 int64_t* sv_out, int64_t* iters_done, int32_t* converged, double* hist);

// rpca_dev, continued on the dense device path (rpca_cb_host with its built-in hooks: full Jacobi SVT + exact stop test
// every iteration, no rank limit) when a single-GPU solve leaves the accelerated kernels -- 512 < min(M,N) <= 2048 with
// a rank estimate above 32, or with hankel=true.  Slower, but the reference has no such limit either.
int rpca_dev_any(tlsq_handle* h, const double* D, int64_t M, int64_t N, const RpcaParams& p, const RpcaOut& o) {
    t_dense_fallback = false;
    const int rc = rpca_dev(h, D, M, N, p, o);
    if (rc == TLSQ_ERR_UNSUPPORTED && t_dense_fallback && h->nranks == 1) {
        t_dense_fallback = false;
        CK(cudaStreamSynchronize(h->stream));
        return rpca_cb_host(h, D, M, N, p, nullptr, nullptr, nullptr, o.A, o.E, o.U, o.S, o.Vt, o.sv, o.iters_done,
                            o.converged, o.hist);
    }
    return rc;
}

// ----------------------------------------------------------------------------------------------------------
// Grassmann averages core (device pointers)
// ----------------------------------------------------------------------------------------------------------
int rpca_ga_dev(tlsq_handle* h, const double* X, int64_t d, int64_t N, int64_t r, const double* q0, double tol,
                int64_t iters, double* Q, int64_t* iters_done, int mu_kind = 0, double mu_p = 0.1) {
    if (d < 1 || N < 1 || r < 1) return set_err(TLSQ_ERR_ARG, "rpca_ga: empty problem");
    if (!X || !q0 || !Q) return set_err(TLSQ_ERR_ARG, "rpca_ga: X, q0 and Q are required");
    if (iters < 1) return set_err(TLSQ_ERR_ARG, "rpca_ga: iters must be >= 1");
    cudaStream_t st = h->stream;
    const int sms = h->sm_count;
    int64_t* L = &h->launches;
    const size_t dn = (size_t)d * N;
    DevBuf bX, bT, bT2, bN2, bS, bQ, bQ2, bQn, bMu, bXs, bSc, bPart;
    CK(bX.alloc(dn * 8, st)); CK(bT.alloc((size_t)(N + 1) * 8, st)); CK(bT2.alloc((size_t)(N + 1) * 8, st));
    CK(bN2.alloc((size_t)N * 8, st));
    CK(bS.alloc((size_t)N * 8, st)); CK(bQ.alloc((size_t)d * 8, st)); CK(bQ2.alloc((size_t)d * 8, st));
    CK(bQn.alloc((size_t)d * 8, st));
    CK(bMu.alloc((size_t)d * 8, st)); CK(bXs.alloc((size_t)N * 8, st)); CK(bSc.alloc(8 * 8, st));
    CK(bPart.alloc(ga_partial_doubles(sms) * 8, st));
    // robust averages over more than kGaRobustMaxN observations: per-row selection (ga_select.cu) instead of a sort
    const bool select = mu_kind != 0 && N > kGaRobustMaxN;
    DevBuf bSel;
    if (select) CK(bSel.alloc(ga_select_bytes(d, N, sms), st));
    void* sel = bSel.p;
    double* Xw = bX.as<double>(); double* n2 = bN2.as<double>();
    double* tb[2] = {bT.as<double>(), bT2.as<double>()};           // dot products: iteration `it` writes tb[it & 1]
    double* s = bS.as<double>(); double* mu = bMu.as<double>();
    double* qb[2] = {bQ.as<double>(), bQ2.as<double>()};            // q ping-pong: the run-ahead iteration must not clobber
    double* qnext = bQn.as<double>();                               // normalised start vector of the next component
    double* xs = bXs.as<double>(); double* sc = bSc.as<double>();   // sc[0] = sumw, sc[1] = ss, sc[2], sc[3] = dq2 slots
    double* part = bPart.as<double>();
    double* hp = h->h_pin;
    const bool no_ahead = getenv("TLSQ_NO_RUNAHEAD") != nullptr;
    CK(cudaMemcpyAsync(Xw, X, dn * 8, cudaMemcpyDeviceToDevice, st));                    // X = copy(X)   :257

    // q = randn(d); q ./= norm(q)   (:286-287) -- the draw comes from the caller
    auto normalise_start = [&](int64_t comp, double* out) -> int {
        CK(cudaMemsetAsync(sc + 1, 0, 8, st));
        CK(launch_vec_sumsq(q0 + comp * d, d, sc + 1, sms, st, L));
        CKR(allreduce(h, sc + 1, 1, kNcclSum));
        CK(launch_vec_scale_rsqrt(q0 + comp * d, sc + 1, d, out, sms, st, L));
        return TLSQ_OK;
    };
    bool head_ready = false;      // n2 and tb[0] of this component already came with the previous component's deflation
    for (int64_t i = 0; i < r; ++i) {                                                    // :263
        int cq = 0;                                                                      // qb[cq] = current q
        if (!head_ready) {
            CK(cudaMemsetAsync(n2, 0, (size_t)N * 8, st));
            CK(launch_ga_sweep(GA_NORMS, Xw, d, N, d, nullptr, nullptr, nullptr, n2, sms, st, L, part));   // :265
            CKR(allreduce(h, n2, (size_t)N, kNcclSum));
            CKR(normalise_start(i, qb[0]));
            CK(cudaMemsetAsync(tb[0], 0, (size_t)(N + 1) * 8, st));
            CK(launch_ga_sweep(GA_DOTS, Xw, d, N, d, qb[0], nullptr, nullptr, tb[0], sms, st, L, part));   // U[:,n]'q  :292
            CKR(allreduce(h, tb[0], (size_t)N, kNcclSum));
        } else {
            CK(cudaMemcpyAsync(qb[0], qnext, (size_t)d * 8, cudaMemcpyDeviceToDevice, st));
        }
        head_ready = false;
        // trimmed mean: the keys X[j,n] / ||x_n|| are fixed until the deflation, so are the rows' kept ranges
        if (select && mu_kind == 1) CK(launch_ga_select(Xw, d, N, d, s, n2, 1, mu_p, sel, nullptr, sms, st, L));
        // One Grassmann iteration on the device (:291-296): signs from the dot products of the previous sweep (tb[(it-1)&1]),
        // one sweep (mu, next dot products into tb[it&1], ||mu||^2), q_new into the OTHER q buffer, ||q_new - q||^2
        // into slot `it & 1`.
        auto enqueue_iteration = [&](int64_t it, int from) -> int {
            const double* tin = tb[(it - 1) & 1];
            double* t = tb[it & 1];
            CK(launch_ga_signs(tin, n2, N, s, sc, st, L));
            CK(cudaMemsetAsync(t, 0, (size_t)(N + 1) * 8, st));
            if (mu_kind == 0) {
                Phase ph(h, TLSQ_PHASE_GA_SWEEP);
                CK(launch_ga_sweep(GA_PASS, Xw, d, N, d, mu, s, sc, t, sms, st, L, part));   // :291-294 in one sweep
            } else {
                // robust entry-wise average (:323-333 / :349-357): a per-row sort over the observations (rows are local
                // to a shard), then ||mu||^2 and the dot products of the NEXT iteration with q = mu/||mu|| -- the sign
                // of u_n'q equals the sign of x_n'mu, so the dots are taken with mu directly
                Phase ph(h, TLSQ_PHASE_GA_SWEEP);
                if (!select) CK(launch_ga_robust(Xw, d, N, d, s, n2, mu_kind, mu_p, mu, sms, st, L));
                else if (mu_kind == 1) CK(launch_ga_trimmed_sweep(Xw, d, N, d, s, n2, mu_p, sel, mu, sms, st, L));
                else CK(launch_ga_select(Xw, d, N, d, s, n2, 2, mu_p, sel, mu, sms, st, L));
                CK(launch_vec_sumsq(mu, d, t + N, sms, st, L));
                CK(launch_ga_sweep(GA_DOTS, Xw, d, N, d, mu, nullptr, nullptr, t, sms, st, L, part));
            }
            CKR(allreduce(h, t, (size_t)(N + 1), kNcclSum));
            double* dq = sc + 2 + (it & 1);
            CK(cudaMemsetAsync(dq, 0, 8, st));
            CK(launch_ga_update(mu, t + N, d, qb[from], qb[from ^ 1], dq, sms, st, L));  // :295-296, 302
            CKR(allreduce(h, dq, 1, kNcclSum));
            CK(cudaMemcpyAsync(hp + (it & 1), dq, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaEventRecord(it & 1 ? h->ev_iter : h->ev_d2h, st));
            return TLSQ_OK;
        };
        // The host only needs ||q_new - q|| to decide when to stop (:298): while it waits for iteration `it`, iteration
        // `it + 1` is already enqueued (run-ahead), so the GPU never idles on the host round trip; if `it` turns out to
        // be the last one the extra iteration is discarded (q and the dot products of iteration `it` live in their own
        // buffers).  Close to the tolerance (last step within 16x) the loop stops running ahead: no wasted sweep.
        int64_t its = 0;
        double dq_prev = 1.0e300;
        CKR(enqueue_iteration(1, cq));
        for (int64_t it = 1; it <= iters; ++it) {                                        // :290
            const int res = cq ^ 1;                     // buffer that iteration `it` writes
            const bool ahead = !no_ahead && it < iters && !(dq_prev < 16.0 * tol);
            if (ahead) CKR(enqueue_iteration(it + 1, res));
            CK(cudaEventSynchronize(it & 1 ? h->ev_iter : h->ev_d2h));
            its = it;
            cq = res;
            dq_prev = sqrt(hp[it & 1]);
            if (dq_prev < tol) break;                                                    // :298
            if (!ahead && it < iters) CKR(enqueue_iteration(it + 1, cq));
        }
        if (iters_done) iters_done[i] = its;
        double* q = qb[cq];
        double* tl = tb[its & 1];                                                        // x_n'mu and ||mu||^2 of the last iteration
        CK(cudaMemcpyAsync(Q + i * d, q, (size_t)d * 8, cudaMemcpyDeviceToDevice, st));  // :269
        if (i + 1 == r) break;                          // X is a private copy: deflating after the last component is moot
        // Xs1 = q'X (:271) = (X'mu) / ||mu|| -- already known from the last sweep, no extra pass over X
        CK(launch_ga_xs(tl, N, xs, st, L));
        CKR(normalise_start(i + 1, qnext));
        CK(cudaMemsetAsync(n2, 0, (size_t)N * 8, st));
        CK(cudaMemsetAsync(tb[0], 0, (size_t)(N + 1) * 8, st));
        // X -= q Xs1 (:272) fused with the norms (:265) and first dot products (:292) of the next component
        cudaError_t fe = launch_ga_deflate_fused(Xw, d, N, d, q, xs, qnext, n2, tb[0], part, sms, st, L);
        if (fe == cudaSuccess) {
            CKR(allreduce(h, n2, (size_t)N, kNcclSum));
            CKR(allreduce(h, tb[0], (size_t)N, kNcclSum));
            head_ready = true;
        } else if (fe != cudaErrorNotSupported) {
            CK(fe);
        } else {
            // the shape does not take the TMA sweep: Xs1 and the deflation as separate passes
            CK(cudaMemsetAsync(xs, 0, (size_t)N * 8, st));
            CK(launch_ga_sweep(GA_DOTS, Xw, d, N, d, q, nullptr, nullptr, xs, sms, st, L, part));  // Xs1 = q'X   :271
            CKR(allreduce(h, xs, (size_t)N, kNcclSum));
            CK(launch_ga_deflate(Xw, d, N, d, q, xs, sms, st, L));                       // :272
        }
    }
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

// ----------------------------------------------------------------------------------------------------------
// lowrankfilter core (device pointers)
// ----------------------------------------------------------------------------------------------------------
int lowrankfilter_dev(tlsq_handle* h, const double* y, int64_t Ns, int64_t n, int64_t lag, RpcaParams p,
                      double* yf, int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist) {
    if (!y || !yf) return set_err(TLSQ_ERR_ARG, "lowrankfilter: y and yf are required");
    if (Ns < 2 || n < 1 || lag < 1) return set_err(TLSQ_ERR_ARG, "lowrankfilter: bad sizes");
    if ((double)n > (double)Ns / 2.0)                                                    // @assert L <= N/2   :79
        return set_err(TLSQ_ERR_ARG, "L has to be less than N/2 = %g", (double)Ns / 2.0);
    if (lag > n) return set_err(TLSQ_ERR_ARG, "lag must be <= L");                       // :80
    const int64_t K = (Ns - n) / lag + 1;                                                // :81
    if (!(p.lambda > 0.0)) p.lambda = 1.0 / sqrt((double)(K > n ? K : n));               // :157
    cudaStream_t st = h->stream;
    // Factored unhankel (lag 1, tall enough for the factored iterate): A is never materialised -- the anti-diagonal
    // sums are taken straight from A_k = clamp(T_k V_k'); sharded runs all-reduce the Ns partial sums.
    {
        int64_t r0, Kl, per, Klast, r0last;
        shard_hankel_rows(K, h->nranks, h->rank, &r0, &Kl);
        shard_hankel_rows(K, h->nranks, 0, &r0last, &per);
        shard_hankel_rows(K, h->nranks, h->nranks - 1, &r0last, &Klast);
        // the decision must be the same on every rank (collectives): test the regular shard and the last one
        auto shard_ok = [&](int64_t rows) {
            return rows >= 1 && (syrk_tma_eligible(reinterpret_cast<const double*>(uintptr_t(256)), rows, n, rows) ||
                                 fused_eligible(MatSrc{y, 1}, true, rows, n));
        };
        if (lag == 1 && K >= n && n <= kEigMaxN && (h->nranks == 1 || shard_ok(per)) && shard_ok(Klast)) {
            CKR(check_rpca_args(Kl, n, p));
            DevBuf bSum;
            CK(bSum.alloc((size_t)Ns * 8, st));
            RpcaOut ol;
            ol.sv = sv; ol.iters_done = iters_done; ol.converged = converged; ol.hist = hist;
            ol.uh_sum = bSum.as<double>(); ol.uh_r0 = r0; ol.uh_Ns = Ns;
            MatSrc srcl{y + r0, 1};
            CKR(rpca_core(h, srcl, true, Kl, n, p, ol));
            CKR(allreduce(h, ol.uh_sum, (size_t)Ns, kNcclSum));
            CK(launch_unhankel_divide_count(ol.uh_sum, K, n, Ns, yf, st, &h->launches));
            CK(cudaStreamSynchronize(st));
            return TLSQ_OK;
        }
    }
    if (h->nranks > 1) {
        // Row-sharded: every rank holds the (small) full signal and works on Hankel rows [r0, r1) through the same
        // implicit index functor; only the n x n Gram, scalars and the anti-diagonal sums are all-reduced.
        if (K < n || n > kEigMaxN)
            return set_err(TLSQ_ERR_UNSUPPORTED, "lowrankfilter (sharded): needs K >= n and n <= %d", kEigMaxN);
        const int64_t base = K / h->nranks, rem = K % h->nranks;
        const int64_t r0 = h->rank * base + (h->rank < rem ? h->rank : rem);
        const int64_t Kl = base + (h->rank < rem ? 1 : 0);
        if (Kl < 1) return set_err(TLSQ_ERR_ARG, "lowrankfilter (sharded): fewer Hankel rows than ranks");
        CKR(check_rpca_args(Kl, n, p));
        DevBuf bAl, bSum;
        CK(bAl.alloc((size_t)Kl * n * 8, st));
        CK(bSum.alloc((size_t)2 * Ns * 8, st));
        RpcaOut ol;
        ol.A = bAl.as<double>(); ol.sv = sv; ol.iters_done = iters_done; ol.converged = converged; ol.hist = hist;
        MatSrc srcl{y + r0 * lag, lag};
        CKR(rpca_core(h, srcl, true, Kl, n, p, ol));
        double* sum = bSum.as<double>();
        double* cnt = sum + Ns;
        CK(cudaMemsetAsync(sum, 0, (size_t)2 * Ns * 8, st));
        CK(launch_unhankel_partial(ol.A, r0, Kl, n, lag, Ns, sum, cnt, st, &h->launches));
        CKR(allreduce(h, sum, (size_t)2 * Ns, kNcclSum));
        CK(launch_unhankel_divide(sum, cnt, Ns, yf, st, &h->launches));
        CK(cudaStreamSynchronize(st));
        return TLSQ_OK;
    }
    DevBuf bA, bH;
    CK(bA.alloc((size_t)K * n * 8, st));
    RpcaOut o;
    o.A = bA.as<double>(); o.sv = sv; o.iters_done = iters_done; o.converged = converged; o.hist = hist;
    if (K >= n) {
        if (n > kEigMaxN)
            return set_err(TLSQ_ERR_UNSUPPORTED, "lowrankfilter: n = %lld exceeds the supported %d", (long long)n,
                           kEigMaxN);
        CKR(check_rpca_args(K, n, p));
        MatSrc src{y, lag};                    // implicit Hankel: H[k,l] = y[k*lag + l], never materialised
        t_dense_fallback = false;
        const int rc = rpca_core(h, src, true, K, n, p, o);
        if (rc == TLSQ_ERR_UNSUPPORTED && t_dense_fallback && h->nranks == 1) {
            // n > 512 and a rank estimate above 32: materialise the embedding, continue on the dense device path
            t_dense_fallback = false;
            CK(cudaStreamSynchronize(st));
            CK(bH.alloc((size_t)K * n * 8, st));
            CK(launch_hankel(y, K, n, lag, bH.as<double>(), st, &h->launches));
            CKR(rpca_cb_host(h, bH.as<double>(), K, n, p, nullptr, nullptr, nullptr, o.A, nullptr, nullptr, nullptr, nullptr,
                             sv, iters_done, converged, hist));
        } else if (rc != TLSQ_OK) {
            return rc;
        }
    } else {
        CK(bH.alloc((size_t)K * n * 8, st));
        CK(launch_hankel(y, K, n, lag, bH.as<double>(), st, &h->launches));
        CKR(rpca_dev_any(h, bH.as<double>(), K, n, p, o));
    }
    CK(launch_unhankel(o.A, K, n, lag, Ns, yf, st, &h->launches));                       // :127
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

// G = X'X of a dense tall matrix (no all-reduce)
int gram_dense(tlsq_handle* h, const double* X, int64_t M, int64_t n, double* G) {
    cudaStream_t st = h->stream;
    DevBuf bP;
    if (syrk_tma_eligible(X, M, n, M)) {
        SyrkPlan sp = syrk_plan(M, n, h->sm_count);
        CK(bP.alloc(sp.partial_bytes, st));
        CK(launch_syrk_tma(X, M, n, M, sp, bP.as<double>(), G, st, &h->launches));
    } else {
        GramPlan plan = gram_plan(M, n, h->sm_count);
        CK(bP.alloc(plan.partial_bytes, st));
        GramSrc gs;
        gs.D = MatSrc{X, M}; gs.A = nullptr; gs.Y = nullptr; gs.A2 = nullptr; gs.ldw = M; gs.M = M; gs.N = n;
        gs.im = 0.0; gs.eps = 0.0; gs.nonnegE = 0;
        CK(launch_gram(gs, GRAM_D, false, plan, bP.as<double>(), G, st, &h->launches));
    }
    return TLSQ_OK;
}

// ----------------------------------------------------------------------------------------------------------
// lowrankfilter, general form (src/robustPCA.jl:119-128): Dch channels (y: Ns x Dch column-major) and the sv > 0
// plain-SSA branch (:123-125).  One channel with sv <= 0 takes the implicit-Hankel path above; everything else
// materialises the K x (n Dch) trajectory matrix (these shapes are small: the multi-channel / SSA uses of the
// reference are test-sized) and reuses rpca_dev / the Gram + Jacobi building blocks.
// ----------------------------------------------------------------------------------------------------------
int lowrankfilter_general_dev(tlsq_handle* h, const double* y, int64_t Ns, int64_t Dch, int64_t n, int64_t lag,
                              int64_t sv_ssa, RpcaParams p, double* yf, int64_t* sv, int64_t* iters_done,
                              int32_t* converged, double* hist) {
    if (Dch == 1 && sv_ssa <= 0)
        return lowrankfilter_dev(h, y, Ns, n, lag, p, yf, sv, iters_done, converged, hist);
    if (!y || !yf) return set_err(TLSQ_ERR_ARG, "lowrankfilter: y and yf are required");
    if (Ns < 2 || n < 1 || lag < 1 || Dch < 1) return set_err(TLSQ_ERR_ARG, "lowrankfilter: bad sizes");
    if ((double)n > (double)Ns / 2.0) return set_err(TLSQ_ERR_ARG, "L has to be less than N/2 = %g", (double)Ns / 2.0);
    if (lag > n) return set_err(TLSQ_ERR_ARG, "lag must be <= L");
    if (h->nranks > 1)
        return set_err(TLSQ_ERR_UNSUPPORTED, "lowrankfilter: multi-channel / sv > 0 forms are single-GPU only");
    cudaStream_t st = h->stream;
    int64_t* L = &h->launches;
    const int64_t K = (Ns - n) / lag + 1, Lc = n * Dch;
    DevBuf bH, bA;
    CK(bH.alloc((size_t)K * Lc * 8, st)); CK(bA.alloc((size_t)K * Lc * 8, st));
    double* H = bH.as<double>(); double* A = bA.as<double>();
    CK(launch_hankel_mc(y, Ns, Dch, K, n, lag, H, st, L));                                // :120
    if (sv_ssa > 0) {
        // s = svd(H); A = U[:, 1:sv] S[1:sv] Vt[1:sv, :]  ==  H V_sv V_sv'  (tall) or  U_sv U_sv' H  (wide)   :124-125
        const bool tall = K >= Lc;
        const int64_t mm = tall ? K : Lc, nn = tall ? Lc : K;
        if (nn > kEigMaxN) return set_err(TLSQ_ERR_UNSUPPORTED, "lowrankfilter(sv>0): min(K, n D) = %lld exceeds %d",
                                          (long long)nn, kEigMaxN);
        int64_t svc = sv_ssa > nn ? nn : sv_ssa;
        DevBuf bT, bG, bV, bLam, bE, bAt;
        const double* X = H;
        if (!tall) {
            CK(bT.alloc((size_t)K * Lc * 8, st));
            CK(launch_transpose(H, K, Lc, bT.as<double>(), st, L));
            X = bT.as<double>();
        }
        CK(bG.alloc((size_t)nn * nn * 8, st)); CK(bV.alloc((size_t)nn * nn * 8, st)); CK(bLam.alloc((size_t)nn * 8, st));
        CKR(gram_dense(h, X, mm, nn, bG.as<double>()));
        CK(bE.alloc(eig_work_doubles((int)nn) * 8, st));
        EigWork ew;
        double* base = bE.as<double>();
        const size_t np = (size_t)nn + 34;
        ew.X0 = base; base += (size_t)nn * nn;
        ew.Xo = base; base += np * nn;
        ew.Vo = base; base += np * nn;
        ew.lam_raw = base; base += np;
        ew.perm = reinterpret_cast<int*>(base); base += nn;
        ew.info = reinterpret_cast<int*>(base);
        CK(launch_eigh(bG.as<double>(), (int)nn, nullptr, ew, bLam.as<double>(), bV.as<double>(), h->sm_count, st, L));
        if (tall) {
            CK(launch_ssa_project(MatSrc{X, mm}, false, mm, nn, bV.as<double>(), (int)svc, A, h->sm_count, st, L));
        } else {
            CK(bAt.alloc((size_t)K * Lc * 8, st));
            CK(launch_ssa_project(MatSrc{X, mm}, false, mm, nn, bV.as<double>(), (int)svc, bAt.as<double>(), h->sm_count,
                                  st, L));
            CK(launch_transpose(bAt.as<double>(), Lc, K, A, st, L));
        }
        if (sv) *sv = svc;
        if (iters_done) *iters_done = 0;
        if (converged) *converged = 1;
        CK(cudaStreamSynchronize(st));       // temporaries above are freed in stream order after this point
    } else {
        if (!(p.lambda > 0.0)) p.lambda = 1.0 / sqrt((double)(K > Lc ? K : Lc));           // :157
        RpcaOut o;
        o.A = A; o.sv = sv; o.iters_done = iters_done; o.converged = converged; o.hist = hist;
        CKR(rpca_dev_any(h, H, K, Lc, p, o));                                             // :122
    }
    if (Dch == 1) CK(launch_unhankel(A, K, n, lag, Ns, yf, st, L));                       // :127
    else CK(launch_unhankel_mc(A, K, n, lag, Ns, Dch, yf, st, L));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}


// ----------------------------------------------------------------------------------------------------------
// rpca with the reference's plugin callables svd / opnorm (src/robustPCA.jl:168-169; used at :177, :193-197, :225).
// A Julia closure reaches this file as a C function pointer; the matrices cross the boundary in HOST memory, so every
// call costs a device->host and a host->device copy: this is the reference's plugin hook, not the fast path.  The
// iterate is dense, every step a plain kernel / GEMM; NULL callables use the built-in device implementations (full
// Jacobi spectrum).  M x N of any orientation with min(M, N) <= kEigMaxN.
// ----------------------------------------------------------------------------------------------------------
struct EigScratch {            // n x n eigen workspace for the helpers below
    DevBuf bG, bV, bLam, bE;
    EigWork ew;
    int n = 0;
    int init(int nn, cudaStream_t st) {
        n = nn;
        CK(bG.alloc((size_t)n * n * 8, st)); CK(bV.alloc((size_t)n * n * 8, st)); CK(bLam.alloc((size_t)n * 8, st));
        CK(bE.alloc(eig_work_doubles(n) * 8, st));
        double* base = bE.as<double>();
        const size_t np = (size_t)n + 34;
        ew.X0 = base; base += (size_t)n * n;
        ew.Xo = base; base += np * n;
        ew.Vo = base; base += np * n;
        ew.lam_raw = base; base += np;
        ew.perm = reinterpret_cast<int*>(base); base += n;
        ew.info = reinterpret_cast<int*>(base);
        return TLSQ_OK;
    }
};

// spectral norm of a dense M x N device matrix (Gram on the short side + full Jacobi); Xt: M x N scratch for wide X
int device_opnorm(tlsq_handle* h, const double* X, int64_t M, int64_t N, double* Xt, EigScratch& es, double* out) {
    cudaStream_t st = h->stream;
    const double* T = X;
    int64_t m = M, n = N;
    if (M < N) { CK(launch_transpose(X, M, N, Xt, st, &h->launches)); T = Xt; m = N; n = M; }
    CKR(gram_dense(h, T, m, n, es.bG.as<double>()));
    CK(launch_eigh(es.bG.as<double>(), (int)n, nullptr, es.ew, es.bLam.as<double>(), es.bV.as<double>(), h->sm_count, st,
                   &h->launches));
    CK(cudaMemcpyAsync(h->h_pin, es.bLam.as<double>(), 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *out = sqrt(h->h_pin[0] > 0.0 ? h->h_pin[0] : 0.0);
    return TLSQ_OK;
}

// thin SVD of a TALL dense device matrix W (M x n, M >= n) to LAPACK accuracy: eigenvectors of the Gram, then the
// CholeskyQR2-style refinement of rpca_core (see there).  Outputs (device, nullable): U M x n, S n, Vt n x n.
int svd_tall_dev(tlsq_handle* h, const double* W, int64_t M, int n, EigScratch& es, double* U, double* S, double* Vt) {
    cudaStream_t st = h->stream;
    int64_t* L = &h->launches;
    DevBuf bC, bB, bK, bV2, bVf, bSc, bSig, bG2;
    CK(bC.alloc((size_t)M * n * 8, st)); CK(bB.alloc((size_t)n * n * 8, st)); CK(bK.alloc((size_t)n * n * 8, st));
    CK(bV2.alloc((size_t)n * n * 8, st)); CK(bVf.alloc((size_t)n * n * 8, st)); CK(bSc.alloc((size_t)n * 8, st));
    CK(bSig.alloc((size_t)n * 8, st)); CK(bG2.alloc((size_t)n * n * 8, st));
    double* G = es.bG.as<double>(); double* V = es.bV.as<double>(); double* lam = es.bLam.as<double>();
    double* sig = bSig.as<double>();
    DevBuf bF, bSvp;
    CK(bF.alloc((size_t)n * 8, st)); CK(bSvp.alloc(16, st));
    CKR(gram_dense(h, W, M, n, G));
    CK(launch_eigh(G, n, nullptr, es.ew, lam, V, h->sm_count, st, L));
    CK(launch_svt_post(lam, n, 0.0, 0, sig, bF.as<double>(), bSvp.as<int>(), st, L));           // sig = sqrt(lam)
    CK(launch_scale_cols_floor(V, sig, n, 1.0e-8, bB.as<double>(), bSc.as<double>(), st, L));
    CK(launch_gemm_any(W, M, n, M, bB.as<double>(), n, bC.as<double>(), st, L));
    CKR(gram_dense(h, bC.as<double>(), M, n, bG2.as<double>()));
    CK(launch_chol_upper(bG2.as<double>(), n, st, L));
    CK(launch_scale_cols_mul(bG2.as<double>(), bSc.as<double>(), n, bK.as<double>(), st, L));
    CK(launch_eigh(bK.as<double>(), n, nullptr, es.ew, sig, bV2.as<double>(), h->sm_count, st, L, nullptr, 1));
    CK(launch_gemm_nn(V, bV2.as<double>(), n, bVf.as<double>(), st, L));
    if (S) CK(cudaMemcpyAsync(S, sig, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
    if (Vt) CK(launch_transpose(bVf.as<double>(), n, n, Vt, st, L));
    if (U) {
        CK(launch_scale_cols_inv(bVf.as<double>(), sig, n, bB.as<double>(), st, L));
        CK(launch_gemm_any(W, M, n, M, bB.as<double>(), n, U, st, L));
    }
    CK(cudaStreamSynchronize(st));        // the temporaries above are released in stream order after this point
    return TLSQ_OK;
}

int rpca_cb_host(tlsq_handle* h, const double* Dh, int64_t M, int64_t N, const RpcaParams& p, tlsq_svd_fn svd_fn,
                 tlsq_opnorm_fn opn_fn, void* user, double* Ah, double* Eh, double* Uh, double* Sh, double* Vth,
                 int64_t* sv_out, int64_t* iters_done, int32_t* converged, double* hist) {
    CKR(check_rpca_args(M, N, p));
    cudaStream_t st = h->stream;
    int64_t* L = &h->launches;
    const int sms = h->sm_count;
    const int64_t d = M < N ? M : N;
    if (d > kEigMaxN) return set_err(TLSQ_ERR_UNSUPPORTED, "rpca: min(M,N) = %lld exceeds the supported %d", (long long)d, kEigMaxN);
    if (h->nranks > 1) return set_err(TLSQ_ERR_UNSUPPORTED, "rpca with user callables is single-GPU (the callables see the whole matrix)");
    const bool tall = M >= N;
    const int n = (int)d;
    const size_t mn = (size_t)M * N;
    const int nonnegA = (p.flags & TLSQ_NONNEG_A) ? 1 : 0, nonnegE = (p.flags & TLSQ_NONNEG_E) ? 1 : 0;
    const int nukeA = (p.flags & TLSQ_NO_NUKE_A) ? 0 : 1;
    const bool hk = (p.flags & TLSQ_HANKEL) != 0;
    DevBuf bD, bA, bE, bY, bZ, bW, bT, bXt, bUs, bVr, bMean, bScal, bSig, bF, bSvp, bB1;
    CK(bD.alloc(mn * 8, st)); CK(bA.alloc(mn * 8, st)); CK(bE.alloc(mn * 8, st)); CK(bY.alloc(mn * 8, st));
    CK(bZ.alloc(mn * 8, st)); CK(bW.alloc(mn * 8, st)); CK(bT.alloc(mn * 8, st)); CK(bXt.alloc(mn * 8, st));
    CK(bUs.alloc((size_t)(M > N ? M : N) * n * 8, st)); CK(bVr.alloc((size_t)n * (M > N ? M : N) * 8, st));
    CK(bMean.alloc((size_t)(M + N) * 8, st)); CK(bScal.alloc(64, st)); CK(bSig.alloc((size_t)n * 8, st));
    CK(bF.alloc((size_t)n * 8, st)); CK(bSvp.alloc(16, st)); CK(bB1.alloc((size_t)n * n * 8, st));
    double* D = bD.as<double>(); double* A = bA.as<double>(); double* E = bE.as<double>(); double* Y = bY.as<double>();
    double* Z = bZ.as<double>(); double* W = bW.as<double>(); double* dscal = bScal.as<double>();
    EigScratch es;
    CKR(es.init(n, st));
    // host staging for the user callables only (none of it exists on the all-device fallback of tlsq_rpca_f64)
    std::vector<double> Zh, Us, Ss, Vts, Usc, Vrc;
    if (svd_fn || opn_fn) Zh.resize(mn);
    if (svd_fn) { Us.resize((size_t)M * n); Ss.resize(n); Vts.resize((size_t)n * N); Usc.resize((size_t)M * n); Vrc.resize((size_t)n * N); }
    int64_t r_user = -1;                     // rank of the last user SVD (-1: the last SVD was the built-in one)
    CK(cudaMemcpyAsync(D, Dh, mn * 8, cudaMemcpyDefault, st));      // host or device pointer (UVA)
    CK(cudaMemsetAsync(A, 0, mn * 8, st));
    CK(cudaMemsetAsync(dscal, 0, 64, st));
    // ---- setup (:174-185) ----
    double norm2 = 0.0;
    if (opn_fn) norm2 = opn_fn(user, Dh, M, N);                                          // opnorm(Y)::RT  :177
    else CKR(device_opnorm(h, D, M, N, bXt.as<double>(), es, &norm2));
    if (!(norm2 > 0.0) || norm2 != norm2) return set_err(TLSQ_ERR_ARG, "rpca: opnorm(D) returned %g", norm2);
    CK(launch_maxabs(MatSrc{D, M}, false, M, N, dscal + 1, sms, st, L));
    CK(cudaMemcpyAsync(h->h_pin, dscal + 1, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const double norminf = h->h_pin[0] / p.lambda;
    const double dual_norm = norm2 > norminf ? norm2 : norminf;
    const double d_norm = norm2;
    double mu = 1.25 / norm2;
    const double mubar = mu * 1.0e7;
    CK(launch_init_ya(MatSrc{D, M}, false, M, N, dual_norm, Y, nullptr, nullptr, 1.0 / mu, p.lambda / mu, nonnegE, sms, st, L));
    int64_t sv = 10, k_done = 0;
    int conv = 0, svp = 0;
    // built-in SVT of the current W (tall orientation T: m x n): A_T = T V_r f V_r'
    auto builtin_svt = [&](double im) -> int {
        const double* T = W;
        int64_t m = M;
        if (!tall) { CK(launch_transpose(W, M, N, bXt.as<double>(), st, L)); T = bXt.as<double>(); m = N; }
        CKR(gram_dense(h, T, m, n, es.bG.as<double>()));
        CK(launch_eigh(es.bG.as<double>(), n, nullptr, es.ew, es.bLam.as<double>(), es.bV.as<double>(), sms, st, L));
        CK(launch_svt_post(es.bLam.as<double>(), n, im, nukeA, bSig.as<double>(), bF.as<double>(), bSvp.as<int>(), st, L));
        CK(cudaMemcpyAsync(h->h_pin, bSvp.as<int>(), 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        memcpy(&svp, h->h_pin, 4);
        if (svp == 0) { CK(cudaMemsetAsync(A, 0, mn * 8, st)); return TLSQ_OK; }
        // B1 = V_r diag(f) (n x svp): scale the leading columns; Ttmp = T B1 (m x svp); A_T = Ttmp V_r'
        CK(launch_scale_cols_mulvec(es.bV.as<double>(), bF.as<double>(), n, svp, bB1.as<double>(), st, L));
        CK(launch_gemm_any(T, m, n, m, bB1.as<double>(), svp, bUs.as<double>(), st, L));
        CK(launch_transpose(es.bV.as<double>(), n, svp, bVr.as<double>(), st, L));       // V_r' : svp x n
        double* AT = tall ? A : bT.as<double>();
        CK(launch_gemm_any(bUs.as<double>(), m, svp, m, bVr.as<double>(), n, AT, st, L));
        if (!tall) CK(launch_transpose(AT, N, M, A, st, L));
        return TLSQ_OK;
    };
    for (int64_t k = 1; k <= p.iters; ++k) {
        const double im = 1.0 / mu, eps = p.lambda / mu;
        CK(launch_compute_e(MatSrc{D, M}, false, M, N, A, Y, im, eps, nonnegE, E, sms, st, L, W));     // :188-192
        if (svd_fn && k > 1) {                                                                       // svd(Z, sv)  :196
            CK(cudaMemcpyAsync(Zh.data(), W, mn * 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            const int64_t r = svd_fn(user, Zh.data(), M, N, sv, Us.data(), Ss.data(), Vts.data());
            if (r < 0 || r > d) return set_err(TLSQ_ERR_ARG, "rpca: the svd callable returned rank %lld (expected 0..%lld)", (long long)r, (long long)d);
            r_user = r;
            svp = 0;
            for (int64_t i = 0; i < r; ++i) svp += (Ss[i] >= im) ? 1 : 0;                            // :198
            if (svp == 0) {
                CK(cudaMemsetAsync(A, 0, mn * 8, st));
            } else {
                // A = U[:,1:svp] diag(S - 1/mu) Vt[1:svp,:]   (:207-208; no shift when nukeA=false :211-212); Vt is r x N
                for (int c = 0; c < svp; ++c) {
                    const double f = nukeA ? Ss[c] - im : Ss[c];
                    for (int64_t i = 0; i < M; ++i) Usc[(size_t)c * M + i] = Us[(size_t)c * M + i] * f;
                }
                for (int64_t j = 0; j < N; ++j)
                    for (int c = 0; c < svp; ++c) Vrc[(size_t)j * svp + c] = Vts[(size_t)j * r + c];
                CK(cudaMemcpyAsync(bUs.as<double>(), Usc.data(), (size_t)M * svp * 8, cudaMemcpyHostToDevice, st));
                CK(cudaMemcpyAsync(bVr.as<double>(), Vrc.data(), (size_t)svp * N * 8, cudaMemcpyHostToDevice, st));
                CK(launch_gemm_any(bUs.as<double>(), M, svp, M, bVr.as<double>(), (int)N, A, st, L));
            }
        } else {
            r_user = -1;
            CKR(builtin_svt(im));                                                                    // svd!(Z)  :194
        }
        sv = svp;                                                                                    // :199-204
        if (sv < 1) sv = 1;
        if (p.maxrank > 0 && sv > p.maxrank) sv = p.maxrank;
        if (hk) {                                                                                    // :214-216
            CK(launch_unhankel(A, M, N, 1, M + N - 1, bMean.as<double>(), st, L));
            CK(launch_soft_hankel_apply(A, M, N, bMean.as<double>(), eps, sms, st, L));
        }
        CK(cudaMemsetAsync(dscal, 0, 8, st));
        CK(launch_dense_update(D, A, E, Y, Z, M, N, mu, nonnegA, dscal, sms, st, L));                // :217-222
        mu = fmin(mu * p.rho, mubar);                                                                // :223
        double cost = 0.0;
        if (opn_fn) {                                                                                // opnorm(Z)  :225
            CK(cudaMemcpyAsync(Zh.data(), Z, mn * 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            cost = opn_fn(user, Zh.data(), M, N) / d_norm;
        } else {
            CKR(device_opnorm(h, Z, M, N, bXt.as<double>(), es, &cost));
            cost /= d_norm;
        }
        if (hist) { hist[3 * (k - 1)] = (double)k; hist[3 * (k - 1) + 1] = (double)svp; hist[3 * (k - 1) + 2] = cost; }
        k_done = k;
        if (cost < p.tol) { conv = 1; break; }                                                       // :228
    }
    if (hk) {                                                                                        // :234-236
        CK(launch_unhankel(E, M, N, 1, M + N - 1, bMean.as<double>(), st, L));
        CK(launch_soft_hankel_apply(E, M, N, bMean.as<double>(), p.lambda / mu, sms, st, L));
    }
    if (Ah) CK(cudaMemcpyAsync(Ah, A, mn * 8, cudaMemcpyDefault, st));
    if (Eh) CK(cudaMemcpyAsync(Eh, E, mn * 8, cudaMemcpyDefault, st));
    CK(cudaStreamSynchronize(st));
    // s: the SVD object of the LAST SVT input (:238) -- the user's, or the built-in one to LAPACK accuracy
    if (Uh || Sh || Vth) {
        if (r_user >= 0) {
            if (Uh) { memset(Uh, 0, (size_t)M * d * 8); memcpy(Uh, Us.data(), (size_t)M * r_user * 8); }
            if (Sh) { memset(Sh, 0, (size_t)d * 8); memcpy(Sh, Ss.data(), (size_t)r_user * 8); }
            if (Vth) {
                memset(Vth, 0, (size_t)d * N * 8);
                for (int64_t j = 0; j < N; ++j)
                    for (int64_t c = 0; c < r_user; ++c) Vth[(size_t)j * d + c] = Vts[(size_t)j * r_user + c];
            }
        } else {
            DevBuf bU, bS, bVt;
            const int64_t m = tall ? M : N;
            CK(bU.alloc((size_t)m * n * 8, st)); CK(bS.alloc((size_t)n * 8, st)); CK(bVt.alloc((size_t)n * n * 8, st));
            const double* T = W;
            if (!tall) { CK(launch_transpose(W, M, N, bXt.as<double>(), st, L)); T = bXt.as<double>(); }
            CKR(svd_tall_dev(h, T, m, n, es, bU.as<double>(), bS.as<double>(), bVt.as<double>()));
            if (Sh) CK(cudaMemcpyAsync(Sh, bS.as<double>(), (size_t)n * 8, cudaMemcpyDefault, st));
            if (tall) {
                if (Uh) CK(cudaMemcpyAsync(Uh, bU.as<double>(), (size_t)M * n * 8, cudaMemcpyDefault, st));
                if (Vth) CK(cudaMemcpyAsync(Vth, bVt.as<double>(), (size_t)n * N * 8, cudaMemcpyDefault, st));
            } else {
                // W' = U_t S V_t'  =>  W = V_t S U_t':  U = V_t (M x d) = (Vt_t)',  Vt = U_t' (d x N)
                if (Uh) { CK(launch_transpose(bVt.as<double>(), n, n, bB1.as<double>(), st, L));
                          CK(cudaMemcpyAsync(Uh, bB1.as<double>(), (size_t)M * n * 8, cudaMemcpyDefault, st)); }
                if (Vth) { CK(launch_transpose(bU.as<double>(), N, n, bT.as<double>(), st, L));
                           CK(cudaMemcpyAsync(Vth, bT.as<double>(), (size_t)n * N * 8, cudaMemcpyDefault, st)); }
            }
            CK(cudaStreamSynchronize(st));
        }
    }
    if (sv_out) *sv_out = sv;
    if (iters_done) *iters_done = k_done;
    if (converged) *converged = conv;
    return TLSQ_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------
extern "C" {

int tlsq_abi_version(void) { return TLSQ_ABI_VERSION; }
const char* tlsq_last_error(void) { return g_err; }

int tlsq_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int tlsq_create(int device, tlsq_handle** out) {
    if (!out) return set_err(TLSQ_ERR_ARG, "tlsq_create: out is NULL");
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        return set_err(TLSQ_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0 || device >= n) return set_err(TLSQ_ERR_ARG, "device %d out of range [0,%d)", device, n);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return set_err(TLSQ_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                       prop.major, prop.minor);
    CK(cudaSetDevice(device));
    tlsq_handle* h = new tlsq_handle();
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    CK(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_iter, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_d2h, cudaEventDisableTiming));
    CK(cudaMallocHost(&h->h_pin, 64 * sizeof(double)));
    // keep freed blocks cached between solves -- in a pool of our own (the default pool's attributes are left alone)
    {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        if (cudaMemPoolCreate(&h->pool, &props) == cudaSuccess) {
            uint64_t thr = UINT64_MAX;
            cudaMemPoolSetAttribute(h->pool, cudaMemPoolAttrReleaseThreshold, &thr);
        } else {
            cudaGetLastError();
            h->pool = nullptr;               // fall back to the default pool, untouched
        }
    }
    *out = h;
    return TLSQ_OK;
}

int tlsq_destroy(tlsq_handle* h) {
    if (!h) return TLSQ_OK;
    cudaSetDevice(h->device);
    if (h->comm && g_nccl.destroy) g_nccl.destroy(h->comm);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->side) cudaStreamDestroy(h->side);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->ev_iter) cudaEventDestroy(h->ev_iter);
    if (h->ev_d2h) cudaEventDestroy(h->ev_d2h);
    if (h->h_pin) cudaFreeHost(h->h_pin);
    if (h->pool) { cudaDeviceSynchronize(); cudaMemPoolDestroy(h->pool); if (t_pool == h->pool) t_pool = nullptr; }
    delete h;
    return TLSQ_OK;
}

int tlsq_set_stream(tlsq_handle* h, void* cuda_stream) {
    if (!h) return set_err(TLSQ_ERR_ARG, "null handle");
    h->stream = (cudaStream_t)cuda_stream;
    return TLSQ_OK;
}

int tlsq_use_own_stream(tlsq_handle* h) {
    if (!h) return set_err(TLSQ_ERR_ARG, "null handle");
    h->stream = h->own_stream;
    return TLSQ_OK;
}

int64_t tlsq_launch_count(const tlsq_handle* h) { return h ? h->launches : 0; }

int tlsq_set_profiling(tlsq_handle* h, int on) {
    if (!h) return set_err(TLSQ_ERR_ARG, "null handle");
    h->prof = on != 0;
    for (int i = 0; i < TLSQ_NUM_PHASES; ++i) { h->phase_ms[i] = 0.0; h->phase_calls[i] = 0; }
    h->spans.clear();
    h->ev_used = 0;
    return TLSQ_OK;
}

int tlsq_get_profile(tlsq_handle* h, double* ms, int64_t* calls) {
    if (!h || !ms || !calls) return set_err(TLSQ_ERR_ARG, "null argument");
    if (cudaSetDevice(h->device) == cudaSuccess && cudaStreamSynchronize(h->stream) == cudaSuccess) prof_collect(h);
    for (int i = 0; i < TLSQ_NUM_PHASES; ++i) { ms[i] = h->phase_ms[i]; calls[i] = h->phase_calls[i]; }
    return TLSQ_OK;
}

int tlsq_comm_unique_id(void* id128) {
    if (!id128) return set_err(TLSQ_ERR_ARG, "id128 is NULL");
    CKR(nccl_load());
    NcclId id;
    int r = g_nccl.get_uid(&id);
    if (r != 0) return set_err(TLSQ_ERR_NCCL, "ncclGetUniqueId failed: %s", g_nccl.errstr ? g_nccl.errstr(r) : "?");
    memcpy(id128, &id, 128);
    return TLSQ_OK;
}

int tlsq_comm_init(tlsq_handle* h, int nranks, int rank, const void* id128) {
    CKR(use_device(h));
    if (nranks < 1 || rank < 0 || rank >= nranks || !id128) return set_err(TLSQ_ERR_ARG, "bad communicator args");
    if (nranks == 1) { h->nranks = 1; h->rank = 0; return TLSQ_OK; }
    CKR(nccl_load());
    NcclId id;
    memcpy(&id, id128, 128);
    int r = g_nccl.init_rank(&h->comm, nranks, id, rank);
    if (r != 0) return set_err(TLSQ_ERR_NCCL, "ncclCommInitRank failed: %s", g_nccl.errstr ? g_nccl.errstr(r) : "?");
    h->nranks = nranks;
    h->rank = rank;
    return TLSQ_OK;
}

// ---- rpca ------------------------------------------------------------------------------------------------
int tlsq_rpca_f64_dev(tlsq_handle* h, const double* D, int64_t M, int64_t N, double lambda, int64_t maxrank,
                      int64_t iters, double tol, double rho, uint32_t flags, double* A, double* E, double* U,
                      double* S, double* Vt, int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist) {
    CKR(use_device(h));
    if (!D) return set_err(TLSQ_ERR_ARG, "rpca: D is NULL");
    RpcaParams p{lambda, tol, rho, maxrank, iters, flags};
    RpcaOut o;
    o.A = A; o.E = E; o.U = U; o.S = S; o.Vt = Vt; o.sv = sv; o.iters_done = iters_done; o.converged = converged;
    o.hist = hist;
    return rpca_dev_any(h, D, M, N, p, o);
}

int tlsq_rpca_f64(tlsq_handle* h, const double* D, int64_t M, int64_t N, double lambda, int64_t maxrank,
                  int64_t iters, double tol, double rho, uint32_t flags, double* A, double* E, double* U, double* S,
                  double* Vt, int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist) {
    CKR(use_device(h));
    if (!D) return set_err(TLSQ_ERR_ARG, "rpca: D is NULL");
    if (M < 1 || N < 1) return set_err(TLSQ_ERR_ARG, "rpca: empty matrix");
    cudaStream_t st = h->stream;
    const size_t mn = (size_t)M * N;
    // thin-SVD width d = min(M_global, N); a row shard (communicator attached) always has M_global >= N (rpca_core)
    const int64_t d = (h->nranks > 1) ? N : (M < N ? M : N);
    DevBuf bD, bA, bE, bU, bS, bVt;
    CK(bD.alloc(mn * 8, st));
    CK(cudaMemcpyAsync(bD.as<double>(), D, mn * 8, cudaMemcpyHostToDevice, st));
    if (A) CK(bA.alloc(mn * 8, st));
    if (E) CK(bE.alloc(mn * 8, st));
    if (U) CK(bU.alloc((size_t)M * d * 8, st));
    if (S) CK(bS.alloc((size_t)d * 8, st));
    if (Vt) CK(bVt.alloc((size_t)d * N * 8, st));
    RpcaParams p{lambda, tol, rho, maxrank, iters, flags};
    RpcaOut o;
    o.A = A ? bA.as<double>() : nullptr; o.E = E ? bE.as<double>() : nullptr; o.U = U ? bU.as<double>() : nullptr;
    o.S = S ? bS.as<double>() : nullptr; o.Vt = Vt ? bVt.as<double>() : nullptr;
    o.sv = sv; o.iters_done = iters_done; o.converged = converged; o.hist = hist;
    bool host_copied = false;                  // A / E went to the host while the SVD was still being computed
    o.hA = A; o.hE = E; o.host_copied = &host_copied;
    t_dense_fallback = false;
    const int rc = rpca_dev(h, bD.as<double>(), M, N, p, o);
    if (rc == TLSQ_ERR_UNSUPPORTED && t_dense_fallback && h->nranks == 1) {
        // 512 < min(M,N) <= 2048 with a rank estimate above 32, or with hankel=true: outside the factored kernels.  Repeat the solve on the
        // dense device path (full Jacobi SVT + exact stop test every iteration: the reference's loop statement by
        // statement, slower but without a rank limit) instead of failing.
        t_dense_fallback = false;
        CK(cudaStreamSynchronize(st));
        bD.release(); bA.release(); bE.release(); bU.release(); bS.release(); bVt.release();
        return rpca_cb_host(h, D, M, N, p, nullptr, nullptr, nullptr, A, E, U, S, Vt, sv, iters_done, converged, hist);
    }
    if (rc != TLSQ_OK) return rc;
    if (A && !host_copied) CK(cudaMemcpyAsync(A, o.A, mn * 8, cudaMemcpyDeviceToHost, st));
    if (E && !host_copied) CK(cudaMemcpyAsync(E, o.E, mn * 8, cudaMemcpyDeviceToHost, st));
    if (U) CK(cudaMemcpyAsync(U, o.U, (size_t)M * d * 8, cudaMemcpyDeviceToHost, st));
    if (S) CK(cudaMemcpyAsync(S, o.S, (size_t)d * 8, cudaMemcpyDeviceToHost, st));
    if (Vt) CK(cudaMemcpyAsync(Vt, o.Vt, (size_t)d * N * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

int tlsq_rpca_cb_f64(tlsq_handle* h, const double* D, int64_t M, int64_t N, double lambda, int64_t maxrank, int64_t iters,
                     double tol, double rho, uint32_t flags, tlsq_svd_fn svd_fn, tlsq_opnorm_fn opnorm_fn, void* user,
                     double* A, double* E, double* U, double* S, double* Vt, int64_t* sv, int64_t* iters_done,
                     int32_t* converged, double* hist) {
    CKR(use_device(h));
    if (!D) return set_err(TLSQ_ERR_ARG, "rpca: D is NULL");
    RpcaParams p{lambda, tol, rho, maxrank, iters, flags};
    return rpca_cb_host(h, D, M, N, p, svd_fn, opnorm_fn, user, A, E, U, S, Vt, sv, iters_done, converged, hist);
}

// ---- lowrankfilter ---------------------------------------------------------------------------------------
int tlsq_lowrankfilter_f64_dev(tlsq_handle* h, const double* y, int64_t Ns, int64_t n, int64_t lag, double lambda,
                               int64_t maxrank, int64_t iters, double tol, double rho, uint32_t flags, double* yf,
                               int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist) {
    CKR(use_device(h));
    RpcaParams p{lambda, tol, rho, maxrank, iters, flags};
    return lowrankfilter_dev(h, y, Ns, n, lag, p, yf, sv, iters_done, converged, hist);
}

int tlsq_lowrankfilter_f64(tlsq_handle* h, const double* y, int64_t Ns, int64_t n, int64_t lag, double lambda,
                           int64_t maxrank, int64_t iters, double tol, double rho, uint32_t flags, double* yf,
                           int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist) {
    CKR(use_device(h));
    if (!y || !yf || Ns < 1) return set_err(TLSQ_ERR_ARG, "lowrankfilter: y and yf are required");
    cudaStream_t st = h->stream;
    DevBuf by, bf;
    CK(by.alloc((size_t)Ns * 8, st)); CK(bf.alloc((size_t)Ns * 8, st));
    CK(cudaMemcpyAsync(by.as<double>(), y, (size_t)Ns * 8, cudaMemcpyHostToDevice, st));
    RpcaParams p{lambda, tol, rho, maxrank, iters, flags};
    CKR(lowrankfilter_dev(h, by.as<double>(), Ns, n, lag, p, bf.as<double>(), sv, iters_done, converged, hist));
    CK(cudaMemcpyAsync(yf, bf.as<double>(), (size_t)Ns * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

// ---- rpca_ga ---------------------------------------------------------------------------------------------
int tlsq_rpca_ga_f64_dev(tlsq_handle* h, const double* X, int64_t d, int64_t N, int64_t r, const double* q0,
                         double tol, int64_t iters, double* Q, int64_t* iters_done) {
    CKR(use_device(h));
    return rpca_ga_dev(h, X, d, N, r, q0, tol, iters, Q, iters_done);
}

int tlsq_rpca_ga_f64(tlsq_handle* h, const double* X, int64_t d, int64_t N, int64_t r, const double* q0, double tol,
                     int64_t iters, double* Q, int64_t* iters_done) {
    CKR(use_device(h));
    if (!X || !q0 || !Q || d < 1 || N < 1 || r < 1) return set_err(TLSQ_ERR_ARG, "rpca_ga: bad arguments");
    cudaStream_t st = h->stream;
    DevBuf bX, bq0, bQ;
    CK(bX.alloc((size_t)d * N * 8, st)); CK(bq0.alloc((size_t)d * r * 8, st)); CK(bQ.alloc((size_t)d * r * 8, st));
    CK(cudaMemcpyAsync(bX.as<double>(), X, (size_t)d * N * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(bq0.as<double>(), q0, (size_t)d * r * 8, cudaMemcpyHostToDevice, st));
    CKR(rpca_ga_dev(h, bX.as<double>(), d, N, r, bq0.as<double>(), tol, iters, bQ.as<double>(), iters_done));
    CK(cudaMemcpyAsync(Q, bQ.as<double>(), (size_t)d * r * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

int tlsq_rpca_ga_mu_f64_dev(tlsq_handle* h, const double* X, int64_t d, int64_t N, int64_t r, const double* q0,
                            double tol, int64_t iters, int mu_kind, double mu_p, double* Q, int64_t* iters_done) {
    CKR(use_device(h));
    if (mu_kind < 0 || mu_kind > 2) return set_err(TLSQ_ERR_ARG, "rpca_ga: mu_kind must be 0 (mean), 1 (trimmed mean) or 2 (median)");
    if (mu_kind == 2 && N < 2) return set_err(TLSQ_ERR_ARG, "rpca_ga: entrywise_median needs at least 2 observations (I[end / 2], src/robustPCA.jl:353)");
    return rpca_ga_dev(h, X, d, N, r, q0, tol, iters, Q, iters_done, mu_kind, mu_p);
}

int tlsq_rpca_ga_mu_f64(tlsq_handle* h, const double* X, int64_t d, int64_t N, int64_t r, const double* q0, double tol,
                        int64_t iters, int mu_kind, double mu_p, double* Q, int64_t* iters_done) {
    CKR(use_device(h));
    if (!X || !q0 || !Q || d < 1 || N < 1 || r < 1) return set_err(TLSQ_ERR_ARG, "rpca_ga: bad arguments");
    if (mu_kind < 0 || mu_kind > 2) return set_err(TLSQ_ERR_ARG, "rpca_ga: mu_kind must be 0 (mean), 1 (trimmed mean) or 2 (median)");
    if (mu_kind == 2 && N < 2) return set_err(TLSQ_ERR_ARG, "rpca_ga: entrywise_median needs at least 2 observations (I[end / 2], src/robustPCA.jl:353)");
    cudaStream_t st = h->stream;
    DevBuf bX, bq0, bQ;
    CK(bX.alloc((size_t)d * N * 8, st)); CK(bq0.alloc((size_t)d * r * 8, st)); CK(bQ.alloc((size_t)d * r * 8, st));
    CK(cudaMemcpyAsync(bX.as<double>(), X, (size_t)d * N * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(bq0.as<double>(), q0, (size_t)d * r * 8, cudaMemcpyHostToDevice, st));
    CKR(rpca_ga_dev(h, bX.as<double>(), d, N, r, bq0.as<double>(), tol, iters, bQ.as<double>(), iters_done, mu_kind, mu_p));
    CK(cudaMemcpyAsync(Q, bQ.as<double>(), (size_t)d * r * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

// ---- hankel / unhankel -----------------------------------------------------------------------------------
int tlsq_hankel_f64(tlsq_handle* h, const double* x, int64_t Ns, int64_t L, int64_t lag, double* H) {
    CKR(use_device(h));
    if (!x || !H || Ns < 1 || L < 1 || lag < 1) return set_err(TLSQ_ERR_ARG, "hankel: bad arguments");
    if ((double)L > (double)Ns / 2.0) return set_err(TLSQ_ERR_ARG, "L has to be less than N/2 = %g", (double)Ns / 2.0);
    if (lag > L) return set_err(TLSQ_ERR_ARG, "lag must be <= L");
    const int64_t K = (Ns - L) / lag + 1;
    cudaStream_t st = h->stream;
    DevBuf bx, bH;
    CK(bx.alloc((size_t)Ns * 8, st)); CK(bH.alloc((size_t)K * L * 8, st));
    CK(cudaMemcpyAsync(bx.as<double>(), x, (size_t)Ns * 8, cudaMemcpyHostToDevice, st));
    CK(launch_hankel(bx.as<double>(), K, L, lag, bH.as<double>(), st, &h->launches));
    CK(cudaMemcpyAsync(H, bH.as<double>(), (size_t)K * L * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

int tlsq_unhankel_f64(tlsq_handle* h, const double* A, int64_t K, int64_t L, int64_t lag, int64_t Ns, double* y) {
    CKR(use_device(h));
    if (!A || !y || K < 1 || L < 1 || lag < 1 || Ns < 1) return set_err(TLSQ_ERR_ARG, "unhankel: bad arguments");
    cudaStream_t st = h->stream;
    DevBuf bA, by;
    CK(bA.alloc((size_t)K * L * 8, st)); CK(by.alloc((size_t)Ns * 8, st));
    CK(cudaMemcpyAsync(bA.as<double>(), A, (size_t)K * L * 8, cudaMemcpyHostToDevice, st));
    CK(launch_unhankel(bA.as<double>(), K, L, lag, Ns, by.as<double>(), st, &h->launches));
    CK(cudaMemcpyAsync(y, by.as<double>(), (size_t)Ns * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

// ---- general forms: channels and the sv > 0 SSA branch ----------------------------------------------------------
int tlsq_lowrankfilter_mc_f64_dev(tlsq_handle* h, const double* y, int64_t Ns, int64_t D, int64_t n, int64_t lag,
                                  int64_t sv_ssa, double lambda, int64_t maxrank, int64_t iters, double tol, double rho,
                                  uint32_t flags, double* yf, int64_t* sv, int64_t* iters_done, int32_t* converged,
                                  double* hist) {
    CKR(use_device(h));
    RpcaParams p{lambda, tol, rho, maxrank, iters, flags};
    return lowrankfilter_general_dev(h, y, Ns, D, n, lag, sv_ssa, p, yf, sv, iters_done, converged, hist);
}

int tlsq_lowrankfilter_mc_f64(tlsq_handle* h, const double* y, int64_t Ns, int64_t D, int64_t n, int64_t lag,
                              int64_t sv_ssa, double lambda, int64_t maxrank, int64_t iters, double tol, double rho,
                              uint32_t flags, double* yf, int64_t* sv, int64_t* iters_done, int32_t* converged,
                              double* hist) {
    CKR(use_device(h));
    if (!y || !yf || Ns < 1 || D < 1) return set_err(TLSQ_ERR_ARG, "lowrankfilter: y and yf are required");
    cudaStream_t st = h->stream;
    DevBuf by, bf;
    CK(by.alloc((size_t)Ns * D * 8, st)); CK(bf.alloc((size_t)Ns * D * 8, st));
    CK(cudaMemcpyAsync(by.as<double>(), y, (size_t)Ns * D * 8, cudaMemcpyHostToDevice, st));
    RpcaParams p{lambda, tol, rho, maxrank, iters, flags};
    CKR(lowrankfilter_general_dev(h, by.as<double>(), Ns, D, n, lag, sv_ssa, p, bf.as<double>(), sv, iters_done,
                                  converged, hist));
    CK(cudaMemcpyAsync(yf, bf.as<double>(), (size_t)Ns * D * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

int tlsq_hankel_mc_f64(tlsq_handle* h, const double* x, int64_t Ns, int64_t D, int64_t L, int64_t lag, double* H) {
    CKR(use_device(h));
    if (!x || !H || Ns < 1 || D < 1 || L < 1 || lag < 1) return set_err(TLSQ_ERR_ARG, "hankel: bad arguments");
    if ((double)L > (double)Ns / 2.0) return set_err(TLSQ_ERR_ARG, "L has to be less than N/2 = %g", (double)Ns / 2.0);
    if (lag > L) return set_err(TLSQ_ERR_ARG, "lag must be <= L");
    const int64_t K = (Ns - L) / lag + 1;
    cudaStream_t st = h->stream;
    DevBuf bx, bH;
    CK(bx.alloc((size_t)Ns * D * 8, st)); CK(bH.alloc((size_t)K * L * D * 8, st));
    CK(cudaMemcpyAsync(bx.as<double>(), x, (size_t)Ns * D * 8, cudaMemcpyHostToDevice, st));
    CK(launch_hankel_mc(bx.as<double>(), Ns, D, K, L, lag, bH.as<double>(), st, &h->launches));
    CK(cudaMemcpyAsync(H, bH.as<double>(), (size_t)K * L * D * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

int tlsq_unhankel_mc_f64(tlsq_handle* h, const double* A, int64_t K, int64_t L, int64_t lag, int64_t Ns, int64_t D,
                         double* y) {
    CKR(use_device(h));
    if (!A || !y || K < 1 || L < 1 || lag < 1 || Ns < 1 || D < 1) return set_err(TLSQ_ERR_ARG, "unhankel: bad arguments");
    cudaStream_t st = h->stream;
    DevBuf bA, by;
    CK(bA.alloc((size_t)K * L * D * 8, st)); CK(by.alloc((size_t)Ns * D * 8, st));
    CK(cudaMemcpyAsync(bA.as<double>(), A, (size_t)K * L * D * 8, cudaMemcpyHostToDevice, st));
    CK(launch_unhankel_mc(bA.as<double>(), K, L, lag, Ns, D, by.as<double>(), st, &h->launches));
    CK(cudaMemcpyAsync(y, by.as<double>(), (size_t)Ns * D * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

// ---- host-only planning helpers (no device needed; exercised by the CPU test-suite) -------------------------------
int tlsq_plan_pipeline(int nranks, const double* votes_sum, int env_fused, int* fused, int* use_w, int* inplace) {
    if (nranks < 1 || !votes_sum || !fused || !use_w || !inplace) return set_err(TLSQ_ERR_ARG, "plan_pipeline: bad arguments");
    const PipelineChoice c = choose_pipeline(nranks, votes_sum, env_fused);
    *fused = c.fused ? 1 : 0; *use_w = c.use_w ? 1 : 0; *inplace = c.inplace_vote ? 1 : 0;
    return TLSQ_OK;
}

int tlsq_plan_fused_strips(uint8_t* tile_row, uint8_t* strip_col) {
    if (!tile_row || !strip_col) return set_err(TLSQ_ERR_ARG, "plan_fused_strips: bad arguments");
    const FusedStripTab t = fused_strip_table();
    memcpy(tile_row, t.row, sizeof(t.row));
    memcpy(strip_col, t.cs, sizeof(t.cs));
    return TLSQ_OK;
}

int tlsq_plan_hankel_shard(int64_t K, int nranks, int rank, int64_t* r0, int64_t* Kl) {
    if (K < 1 || nranks < 1 || rank < 0 || rank >= nranks || !r0 || !Kl) return set_err(TLSQ_ERR_ARG, "plan_hankel_shard: bad arguments");
    shard_hankel_rows(K, nranks, rank, r0, Kl);
    return TLSQ_OK;
}

// ---- building blocks -------------------------------------------------------------------------------------
int tlsq_gram_f64_dev(tlsq_handle* h, const double* X, int64_t M, int64_t n, double* G) {
    CKR(use_device(h));
    if (!X || !G || M < 1 || n < 1) return set_err(TLSQ_ERR_ARG, "gram: bad arguments");
    cudaStream_t st = h->stream;
    DevBuf bP;
    if (syrk_tma_eligible(X, M, n, M)) {
        SyrkPlan sp = syrk_plan(M, n, h->sm_count);
        CK(bP.alloc(sp.partial_bytes, st));
        CK(launch_syrk_tma(X, M, n, M, sp, bP.as<double>(), G, st, &h->launches));
    } else {
        GramPlan plan = gram_plan(M, n, h->sm_count);
        CK(bP.alloc(plan.partial_bytes, st));
        GramSrc gs;
        gs.D = MatSrc{X, M}; gs.A = nullptr; gs.Y = nullptr; gs.A2 = nullptr; gs.ldw = M; gs.M = M; gs.N = n;
        gs.im = 0.0; gs.eps = 0.0; gs.nonnegE = 0;
        CK(launch_gram(gs, GRAM_D, false, plan, bP.as<double>(), G, st, &h->launches));
    }
    CKR(allreduce(h, G, (size_t)n * n, kNcclSum));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

int tlsq_eigh_f64_dev(tlsq_handle* h, const double* G, int64_t n, double* lam, double* V) {
    CKR(use_device(h));
    if (!G || !lam || !V || n < 1) return set_err(TLSQ_ERR_ARG, "eigh: bad arguments");
    if (n > kEigMaxN) return set_err(TLSQ_ERR_UNSUPPORTED, "eigh: n = %lld exceeds %d", (long long)n, kEigMaxN);
    cudaStream_t st = h->stream;
    DevBuf bE;
    CK(bE.alloc(eig_work_doubles((int)n) * 8, st));
    EigWork ew;
    double* base = bE.as<double>();
    const size_t np = (size_t)n + 34;
    ew.X0 = base; base += (size_t)n * n;
    ew.Xo = base; base += np * n;
    ew.Vo = base; base += np * n;
    ew.lam_raw = base; base += np;
    ew.perm = reinterpret_cast<int*>(base); base += n;
    ew.info = reinterpret_cast<int*>(base);
    CK(launch_eigh(G, (int)n, nullptr, ew, lam, V, h->sm_count, st, &h->launches));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

int tlsq_robust_average_f64_dev(tlsq_handle* h, const double* U, int64_t d, int64_t N, const double* w, int kind,
                                double P, double* s) {
    if (!h) {
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
            cudaGetLastError();
            return set_err(TLSQ_ERR_NO_DEVICE, "no CUDA device available (this library has no CPU fallback)");
        }
    }
    CKR(use_device(h));
    if (!U || !w || !s || d < 1 || N < 1) return set_err(TLSQ_ERR_ARG, "robust_average: bad arguments");
    if (kind != 1 && kind != 2) return set_err(TLSQ_ERR_ARG, "robust_average: kind must be 1 (trimmed mean) or 2 (median)");
    if (kind == 1 && !(P >= 0.0 && P <= 1.0)) return set_err(TLSQ_ERR_ARG, "robust_average: P must lie in [0, 1]");
    if (N > (int64_t)0xffffffffLL) return set_err(TLSQ_ERR_UNSUPPORTED, "robust_average: more than 2^32 - 1 observations");
    cudaStream_t st = h->stream;
    DevBuf bW;
    CK(bW.alloc(ga_select_bytes(d, N, h->sm_count), st));
    CK(launch_ga_select(U, d, N, d, w, nullptr, kind, P, bW.p, s, h->sm_count, st, &h->launches));
    if (kind == 1) CK(launch_ga_trimmed_sweep(U, d, N, d, w, nullptr, P, bW.p, s, h->sm_count, st, &h->launches));
    CK(cudaStreamSynchronize(st));
    return TLSQ_OK;
}

}  // extern "C"
