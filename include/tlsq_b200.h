/*
 * tlsq_b200.h -- C ABI of libtlsq_b200.so: the B200-native (sm_100a) robust-PCA hot path of
 * baggepinnen/TotalLeastSquares.jl (rpca / rpca_ga / lowrankfilter and their hankel helpers).
 *
 * This is the drop-in boundary: the entry points below are exactly what a Julia `ccall` shim for
 * `rpca`, `rpca_ga`, `lowrankfilter`, `hankel`, `unhankel` binds (see INTEGRATION.md and
 * totalleastsquares.jl_b200/julia/TotalLeastSquaresB200.jl).  Reference citations (file:line) are relative to
 * the reference repository root.
 *
 * Conventions
 *  - All matrices are dense FP64, COLUMN-MAJOR (Julia layout), leading dimension == number of rows.
 *  - Dimensions are int64_t.  Inputs are never modified (reference: Y = copy(D) src/robustPCA.jl:176,
 *    X = copy(X) :257).  Outputs are caller-allocated; an output pointer may be NULL to skip it.
 *  - `*_f64`      : HOST pointers; the library stages data through device memory (H2D/D2H inside the call).
 *    `*_f64_dev`  : DEVICE pointers on the handle's device; work is enqueued on the handle's stream and the
 *                   call returns after the solve finished (it synchronises the stream).
 *  - Every function returns an int status (TLSQ_OK == 0); tlsq_last_error() gives a thread-local message.
 *    The library never throws, never calls back, and has NO CPU fallback: without a usable sm_100 device every
 *    compute entry point fails with TLSQ_ERR_NO_DEVICE.
 *  - Multi-GPU: one process (or thread) per GPU.  Each rank creates its own handle, joins a communicator with
 *    tlsq_comm_init, and passes its CONTIGUOUS ROW SHARD (rows [r0, r1) of the matrix; for rpca_ga the d
 *    dimension is the sharded one).  Only n x n Gram matrices, length-N vectors and scalars are all-reduced
 *    (NCCL); data rows never move.
 */
#ifndef TLSQ_B200_H
#define TLSQ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TLSQ_ABI_VERSION 1

/* status codes */
#define TLSQ_OK               0
#define TLSQ_ERR_ARG          1   /* invalid argument (dimension, NULL pointer, hankel asserts :79-80) */
#define TLSQ_ERR_NO_DEVICE    2   /* no CUDA device / not sm_100: there is no CPU fallback            */
#define TLSQ_ERR_CUDA         3   /* CUDA runtime error                                               */
#define TLSQ_ERR_NCCL         4   /* NCCL error or libnccl not loadable                               */
#define TLSQ_ERR_UNSUPPORTED  5   /* feature outside the accelerated path (see DESIGN.md, scope)      */
#define TLSQ_ERR_NOMEM        6   /* device allocation failed                                         */

/* rpca flag bits (reference kwargs, src/robustPCA.jl:162-166) */
#define TLSQ_NONNEG_A     (1u << 0)  /* nonnegA=true  (:217-219)                                   */
#define TLSQ_NONNEG_E     (1u << 1)  /* nonnegE=true  (:189-191)                                   */
#define TLSQ_HANKEL       (1u << 2)  /* hankel=true   (:214-216,234-236)  single GPU only          */
#define TLSQ_NO_NUKE_A    (1u << 3)  /* nukeA=false   (:209-213)                                   */
#define TLSQ_EXACT_COST   (1u << 4)  /* evaluate opnorm(Z) exactly every iteration (needed only to print the
                                        verbose cost, :226); otherwise the stop test uses Frobenius brackets and
                                        falls back to the exact spectral norm only when they do not decide */

typedef struct tlsq_handle tlsq_handle;

/* ---- library / handle ------------------------------------------------------------------------------------- */
int         tlsq_abi_version(void);
const char* tlsq_last_error(void);
/* number of usable CUDA devices (0 if none; never fails) */
int         tlsq_device_count(void);
/* create a solver context on CUDA device `device` (owns a stream, workspaces, optional NCCL communicator) */
int         tlsq_create(int device, tlsq_handle** out);
int         tlsq_destroy(tlsq_handle* h);
/* enqueue all work of this handle on an externally owned cudaStream_t (NULL == the CUDA default stream, e.g.
 * torch's current stream so that the caller's producers/consumers and CUDA events are ordered with the solve) */
int         tlsq_set_stream(tlsq_handle* h, void* cuda_stream);
/* go back to the handle's own non-blocking stream (the default after tlsq_create) */
int         tlsq_use_own_stream(tlsq_handle* h);
/* number of kernels launched through this handle since creation (bench.py's gpu_launches) */
int64_t     tlsq_launch_count(const tlsq_handle* h);

/* optional device-side phase timing (CUDA events on the solve stream; off by default).  tlsq_set_profiling resets
 * the accumulators; tlsq_get_profile returns accumulated milliseconds and span counts per phase. */
#define TLSQ_NUM_PHASES        9
#define TLSQ_PHASE_GRAM        0   /* DMMA Gram of the SVT input (+ deterministic reduce)            */
#define TLSQ_PHASE_EIG         1   /* n x n Jacobi eigensolver (+ warm-start GEMM, sort, shrink)     */
#define TLSQ_PHASE_EPILOGUE    2   /* fused E / W / A / Z / Y pass                                    */
#define TLSQ_PHASE_EXACT_COST  3   /* Gram of Z + eigensolver when the Frobenius bracket is undecided */
#define TLSQ_PHASE_INIT        4   /* opnorm(D), max|D|, Y = D/dual                                   */
#define TLSQ_PHASE_FINALIZE    5   /* E, U, S, Vt outputs                                             */
#define TLSQ_PHASE_ALLREDUCE   6   /* NCCL all-reduces                                                */
#define TLSQ_PHASE_GA_SWEEP    7   /* Grassmann-average streaming sweep                               */
#define TLSQ_PHASE_FUSED       8   /* one-pass ALM step: epilogue of iteration k + Gram of iteration k+1 */
int tlsq_set_profiling(tlsq_handle* h, int on);
int tlsq_get_profile(tlsq_handle* h, double* ms, int64_t* calls);

/* ---- multi-GPU (row-sharded) ------------------------------------------------------------------------------ */
/* fill a 128-byte NCCL unique id (rank 0 calls this and broadcasts the bytes to the other ranks) */
int tlsq_comm_unique_id(void* id128);
/* join a communicator of `nranks` ranks as `rank`; afterwards every solve on this handle is collective */
int tlsq_comm_init(tlsq_handle* h, int nranks, int rank, const void* id128);

/* ---- rpca : replaces rpca(D; kwargs...) src/robustPCA.jl:156-239 ------------------------------------------
 * D      : M x N (this rank's row shard when a communicator is attached)
 * lambda : reference default 1/sqrt(max(M,N)) (:157) is applied by the CALLER (global M!)
 * maxrank: <=0 means typemax(Int) (:158); only clamps the returned sv (:204)
 * iters, tol, rho : :159-161        flags : TLSQ_* bits above
 * outputs (each may be NULL):
 *   A, E   : M x N                                  (:238)
 *   U,S,Vt : thin SVD of the LAST SVT input matrix  (:194,238)  U: M x d, S: d, Vt: d x N, d = min(Mglobal,N)
 *   sv     : estimated rank (:204)       iters_done : number of ALM iterations executed
 *   hist   : iters x 3 doubles, row k-1 = (k, svp, cost) (cost is the exact opnorm ratio when it was evaluated,
 *            otherwise the Frobenius upper bound with a negative sign)
 * returns TLSQ_OK also when `iters` was reached without convergence (the reference only warns, :232);
 * *converged tells the shim whether to emit that warning. */
int tlsq_rpca_f64(tlsq_handle* h, const double* D, int64_t M, int64_t N,
                  double lambda, int64_t maxrank, int64_t iters, double tol, double rho, uint32_t flags,
                  double* A, double* E, double* U, double* S, double* Vt,
                  int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist);
int tlsq_rpca_f64_dev(tlsq_handle* h, const double* D, int64_t M, int64_t N,
                      double lambda, int64_t maxrank, int64_t iters, double tol, double rho, uint32_t flags,
                      double* A, double* E, double* U, double* S, double* Vt,
                      int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist);

/* ---- rpca with the reference's plugin callables `svd` / `opnorm` (src/robustPCA.jl:168-169; used at :177, :193-197,
 * :225; reference test test/runtests.jl:384-398).  A Julia closure reaches the library as a C function pointer
 * (@cfunction) plus an opaque `user` pointer.  The matrices cross the boundary in HOST memory (column-major), so every
 * call costs a device->host and a host->device copy: this is the reference's plugin hook, not the fast path.  NULL
 * selects the built-in device implementation.  Single GPU, host pointers, any orientation, min(M,N) <= 4096.
 *  svd_fn   : thin or truncated SVD of Z (M x N): fill U (M x r, column-major), S (r, descending), Vt (r x N, leading
 *             dimension r) with 0 <= r <= min(M,N) and return r (< 0: error).  Called for k >= 2 with the current `sv`
 *             like the reference's svd(Z, sv) (:196); the first iteration always uses the built-in SVD (:193-194).
 *  opnorm_fn: returns (an estimate of) ||Z||_2 (:177, :225).
 * Outputs as tlsq_rpca_f64; when the last SVD came from svd_fn with r < d the remaining columns / entries of U, S, Vt
 * are zero. */
typedef int64_t (*tlsq_svd_fn)(void* user, const double* Z, int64_t M, int64_t N, int64_t sv,
                               double* U, double* S, double* Vt);
typedef double  (*tlsq_opnorm_fn)(void* user, const double* Z, int64_t M, int64_t N);
int tlsq_rpca_cb_f64(tlsq_handle* h, const double* D, int64_t M, int64_t N,
                     double lambda, int64_t maxrank, int64_t iters, double tol, double rho, uint32_t flags,
                     tlsq_svd_fn svd_fn, tlsq_opnorm_fn opnorm_fn, void* user,
                     double* A, double* E, double* U, double* S, double* Vt,
                     int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist);

/* ---- lowrankfilter : replaces lowrankfilter(y, n; lag=1, sv=0, tol=1e-3, kwargs...) src/robustPCA.jl:119-128
 * for a single channel.  The K x n Hankel embedding (K = (Ns-n)/lag+1, :81) is indexed implicitly from y and is
 * never materialised; the result is the anti-diagonal average of the low-rank part (:127 -> :28-39, :53-68).
 * lambda <= 0 selects the reference default 1/sqrt(max(K,n)).  yf: Ns doubles.                                 */
int tlsq_lowrankfilter_f64(tlsq_handle* h, const double* y, int64_t Ns, int64_t n, int64_t lag,
                           double lambda, int64_t maxrank, int64_t iters, double tol, double rho, uint32_t flags,
                           double* yf, int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist);
int tlsq_lowrankfilter_f64_dev(tlsq_handle* h, const double* y, int64_t Ns, int64_t n, int64_t lag,
                               double lambda, int64_t maxrank, int64_t iters, double tol, double rho, uint32_t flags,
                               double* yf, int64_t* sv, int64_t* iters_done, int32_t* converged, double* hist);

/* ---- rpca_ga : replaces rpca_ga(X, r, U; tol, iters) src/robustPCA.jl:255-306 with the default average mu!
 * (:308-316).  X: d x N, columns are observations (this rank's ROW shard of the d dimension when sharded).
 * q0: d x r start vectors -- column i is the randn(d) the reference draws for component i (:286); the shim draws
 * them so the global-RNG order is preserved.  Q: d x r.  iters_done: r entries (may be NULL).                  */
int tlsq_rpca_ga_f64(tlsq_handle* h, const double* X, int64_t d, int64_t N, int64_t r, const double* q0,
                     double tol, int64_t iters, double* Q, int64_t* iters_done);
int tlsq_rpca_ga_f64_dev(tlsq_handle* h, const double* X, int64_t d, int64_t N, int64_t r, const double* q0,
                         double tol, int64_t iters, double* Q, int64_t* iters_done);

/* rpca_ga with the reference's pluggable robust averages (keyword mu, :255,294): mu_kind 0 = mu! (:308-316),
 * 1 = entrywise_trimmed_mean(s, w, U, P = mu_p) (:323-333), 2 = entrywise_median (:349-357), for any number N of
 * observations: a per-row sort up to 16384 observations, per-row radix selection over streaming sweeps of X beyond.
 * Rows may be sharded like tlsq_rpca_ga_f64.                                                                        */
int tlsq_rpca_ga_mu_f64(tlsq_handle* h, const double* X, int64_t d, int64_t N, int64_t r, const double* q0,
                        double tol, int64_t iters, int mu_kind, double mu_p, double* Q, int64_t* iters_done);
int tlsq_rpca_ga_mu_f64_dev(tlsq_handle* h, const double* X, int64_t d, int64_t N, int64_t r, const double* q0,
                            double tol, int64_t iters, int mu_kind, double mu_p, double* Q, int64_t* iters_done);

/* ---- hankel / unhankel : src/robustPCA.jl:76-92 and :28-39,53-68 (single channel, D == 1) ------------------ */
/* H: K x L with K = (Ns-L)/lag+1;  H[k,l] = x[k*lag + l]  (0-based).  Fails with TLSQ_ERR_ARG when the
 * reference's asserts (L <= Ns/2, lag <= L) fail.                                                               */
int tlsq_hankel_f64(tlsq_handle* h, const double* x, int64_t Ns, int64_t L, int64_t lag, double* H);
/* y: Ns samples; y[t] = mean of all A[k,l] with k*lag + l == t (0 where no entry maps to t, :66)              */
int tlsq_unhankel_f64(tlsq_handle* h, const double* A, int64_t K, int64_t L, int64_t lag, int64_t Ns, double* y);

/* ---- general forms of the three functions above: D channels (x / y: Ns x D column-major; the trajectory matrix is
 * K x (L D) with H[k, l D + d] = x[k lag + l, d], src/robustPCA.jl:83-90; unhankel :53-68) and the sv > 0 plain-SSA
 * branch of lowrankfilter (A = U[:,1:sv] S[1:sv] Vt[1:sv,:] of svd(H), :123-125; sv_ssa <= 0 selects rpca).
 * D == 1 with sv_ssa <= 0 is forwarded to the implicit-Hankel path above; the other cases materialise H
 * (single GPU).                                                                                                  */
int tlsq_lowrankfilter_mc_f64(tlsq_handle* h, const double* y, int64_t Ns, int64_t D, int64_t n, int64_t lag,
                              int64_t sv_ssa, double lambda, int64_t maxrank, int64_t iters, double tol, double rho,
                              uint32_t flags, double* yf, int64_t* sv, int64_t* iters_done, int32_t* converged,
                              double* hist);
int tlsq_lowrankfilter_mc_f64_dev(tlsq_handle* h, const double* y, int64_t Ns, int64_t D, int64_t n, int64_t lag,
                                  int64_t sv_ssa, double lambda, int64_t maxrank, int64_t iters, double tol, double rho,
                                  uint32_t flags, double* yf, int64_t* sv, int64_t* iters_done, int32_t* converged,
                                  double* hist);
int tlsq_hankel_mc_f64(tlsq_handle* h, const double* x, int64_t Ns, int64_t D, int64_t L, int64_t lag, double* H);
int tlsq_unhankel_mc_f64(tlsq_handle* h, const double* A, int64_t K, int64_t L, int64_t lag, int64_t Ns, int64_t D,
                         double* y);

/* ---- host-only planning helpers (no device needed) ----------------------------------------------------------------
 * tlsq_plan_pipeline: the per-iteration pipeline every rank of a sharded solve derives from the rank-summed votes
 *   votes_sum = sum over ranks of {can run the two-kernel pipeline, can run the one-pass kernel, wants the one-pass
 *   kernel for memory, wants Y in place}; env_fused = -1 (unset) / 0 / 1 mirrors TLSQ_FUSED.
 * tlsq_plan_hankel_shard: rows [r0, r0 + Kl) of the K Hankel rows that `rank` owns in a sharded lowrankfilter.
 * tlsq_plan_syrk: the CTA split of the TMA SYRK (G = X'X, X: M x N, 1 <= N <= 4096) on a device with sm_count SMs.
 *   Upper-triangular 128 x 128 blocks b = 0 .. nblk-1 in row order (bi <= bj); block b runs on CTAs
 *   [cta_begin[b], cta_begin[b+1]), nsplit_blk[b] of them, and sums into partial slots [part_off[b], +nsplit_blk[b]).
 *   nsplit_blk and part_off need nb (nb + 1) / 2 entries with nb = ceil(N / 128), cta_begin one more.              */
int tlsq_plan_pipeline(int nranks, const double* votes_sum, int env_fused, int* fused, int* use_w, int* inplace);
int tlsq_plan_hankel_shard(int64_t K, int nranks, int rank, int64_t* r0, int64_t* Kl);
int tlsq_plan_syrk(int64_t M, int64_t N, int sm_count, int* nblk, int* ncta, int* nsplit_blk, int* cta_begin,
                   int* part_off, int64_t* partial_bytes);
/* work split of the one-pass kernel's 256 x 256 Gram: tile_row / strip_col [2 CTAs][8 warps][9 strips] -- strip s of
 * warp w of CTA r is rows [32 tile_row, +32) x columns [8 strip_col, +8) of the upper triangle                      */
int tlsq_plan_fused_strips(uint8_t* tile_row, uint8_t* strip_col);

/* ---- building blocks exposed for tests and profiling (device pointers) ------------------------------------- */
/* G (n x n, column-major) = X' X for X: M x n column-major, via the FP64 tensor-core (DMMA) SYRK kernel       */
int tlsq_gram_f64_dev(tlsq_handle* h, const double* X, int64_t M, int64_t n, double* G);
/* eigen-decomposition of a symmetric PSD n x n matrix (one-sided Jacobi): lam sorted descending, V columns     */
int tlsq_eigh_f64_dev(tlsq_handle* h, const double* G, int64_t n, double* lam, double* V);
/* s (length d) = the reference's robust average mu(s, w, U) of U (d x N, column-major) with weights w (length N):
 * kind 1 = entrywise_trimmed_mean with fraction P (:323-333), kind 2 = entrywise_median (:349-357; for N = 1 the
 * single entry).  Always takes the per-row radix selection kernels that rpca_ga uses beyond 16384 observations.     */
int tlsq_robust_average_f64_dev(tlsq_handle* h, const double* U, int64_t d, int64_t N, const double* w, int kind,
                                double P, double* s);

#ifdef __cplusplus
}
#endif
#endif /* TLSQ_B200_H */
