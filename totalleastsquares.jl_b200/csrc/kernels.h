// kernels.h -- internal launcher interface between the host solver (solver.cu) and the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace tlsq {

// ----------------------------------------------------------------------------------------------------
// Gram (SYRK) pass: G = W'W where W is formed on the fly per element.
// ----------------------------------------------------------------------------------------------------
enum GramMode : int {
    GRAM_D = 0,   // W = D                                  (opnorm(D), src/robustPCA.jl:177)
    GRAM_W = 1,   // W = D - E + Y/mu, E = soft_th(...)     (SVT input, :188-194)
    GRAM_Z = 2    // W = Z = D - A_new - E                  (exact stop test opnorm(Z), :221,225)
};

struct GramSrc {
    MatSrc D;            // dense matrix or implicit Hankel signal
    const double* A;     // A_{k-1}  (modes W, Z)   ld = ldw
    const double* Y;     // Y_{k-1}  (modes W, Z)
    const double* A2;    // A_k      (mode Z)
    int64_t ldw;         // leading dimension of A / Y / A2
    int64_t M, N;
    double im, eps;      // 1/mu, lambda/mu
    int nonnegE;
};

constexpr int kGramBlk = 64;   // output block edge handled by one CTA
constexpr int kGramRows = 32;  // rows (K dimension) per smem tile

// number of upper-triangular blocks / CTA split over rows chosen by the launcher
struct GramPlan { int nb; int nblk; int nsplit; int ntiles; size_t partial_bytes; };
GramPlan gram_plan(int64_t M, int64_t N, int sm_count);
// partial: workspace of plan.partial_bytes; G: N x N (ld N), full symmetric
cudaError_t launch_gram(const GramSrc& s, GramMode mode, bool hankel, const GramPlan& plan, double* partial,
                        double* G, cudaStream_t st, int64_t* launches);

cudaError_t launch_gram_reduce(const double* partial, int nsplit, int nblk, int nb, int B, int N, double* G,
                               cudaStream_t st);

// TMA-fed SYRK for a materialised dense X (syrk_tma.cu): 128 x 128 blocks, 16-row boxes, 4-stage mbarrier ring
constexpr int kSyrkBlk = 128;
constexpr int kEigMaxN = 2048;              // largest min(M, N): 16 x 16 blocks of 128 columns
constexpr int kEigSmallN = 512;             // up to here: shared-memory / register-resident eigen kernels (eig.cu, eig_fast.cu)
constexpr int kSyrkMaxBlk = 136;            // upper-triangular 128-blocks at N = 2048
struct SyrkPlan {
    int nb, nblk, nsplit, ntiles, ncta;     // 128-blocks per dimension, upper-triangular blocks, -, 32-row tiles, CTAs
    int nsplit_blk[kSyrkMaxBlk];            // row splits (CTAs) of every block, proportional to its cost
    int cta_begin[kSyrkMaxBlk + 1];         // first CTA of every block
    int part_off[kSyrkMaxBlk];              // first partial slot of every block
    size_t partial_bytes;
};
bool syrk_tma_eligible(const double* X, int64_t M, int64_t N, int64_t ld);
SyrkPlan syrk_plan(int64_t M, int64_t N, int sm_count);
cudaError_t launch_syrk_tma(const double* X, int64_t M, int64_t N, int64_t ld, const SyrkPlan& plan, double* partial,
                            double* G, cudaStream_t st, int64_t* launches);

// ----------------------------------------------------------------------------------------------------
// Small symmetric eigenproblem (n <= 512): one-sided Jacobi with warp-shuffle rotations.
// ----------------------------------------------------------------------------------------------------
struct EigWork {       // all device pointers, sized for n (see eig_work_bytes)
    double* X0;        // n x n    G * V0
    double* Xo;        // npad x n rotated columns (X part)
    double* Vo;        // npad x n rotated columns (V part)
    double* lam_raw;   // npad
    int*    perm;      // n
    int*    info;      // [0] sweeps done, [1] rotations in last sweep, [2..] per-sweep counters (64)
};
size_t eig_work_doubles(int n);
// Eigen-decomposition of symmetric PSD G (n x n, ld n).  If V0 != nullptr it must hold an orthogonal n x n
// warm-start basis (previous eigenvectors).  Outputs: lam (n, descending), Vs (n x n sorted eigenvector columns).
// Vs may alias V0.
// run_flag (optional, device): the whole decomposition is skipped on the device when run_flag[1] == 0.
// svd_mode != 0: G is a GENERAL square matrix K; its columns are orthogonalised (K V = U S): lam = singular values
// (descending), Vs = right singular vectors.
cudaError_t launch_eigh(const double* G, int n, const double* V0, EigWork w, double* lam, double* Vs,
                        int sm_count, cudaStream_t st, int64_t* launches, const int* run_flag = nullptr,
                        int svd_mode = 0);
// in-place upper Cholesky factor of an n x n SPD matrix (single CTA; deflates pivots that lost all their digits)
cudaError_t launch_chol_upper(double* R, int n, cudaStream_t st, int64_t* launches);
// B[:, c] = V[:, c] / max(sigma_c, floor_rel * sigma_0), sc_out[c] = that scale;   K[:, c] = R[:, c] * sc[c]
cudaError_t launch_scale_cols_floor(const double* V, const double* sigma, int n, double floor_rel, double* B,
                                    double* sc_out, cudaStream_t st, int64_t* launches);
cudaError_t launch_scale_cols_mul(const double* R, const double* sc, int n, double* K, cudaStream_t st,
                                  int64_t* launches);
// B[:, c] = V[:, c] * f[c], c < cols   (n rows)
cudaError_t launch_scale_cols_mulvec(const double* V, const double* f, int n, int cols, double* B, cudaStream_t st,
                                     int64_t* launches);
// C = A B for n x n column-major matrices
cudaError_t launch_gemm_nn(const double* A, const double* B, int n, double* C, cudaStream_t st, int64_t* launches);

// Fast path (eig_fast.cu, 64 < n <= 512; 16-column block only above n = 256): warm-started block subspace iteration for the dominant eigenpairs +
// a rigorous certificate of the count #{sigma >= tau}.  flags[1] != 0 afterwards means "fall back to launch_eigh".
struct EigFastWork {
    double* Qb;      // n x 32 warm-start basis carried between ALM iterations
    double* Qwork;   // n x 32 working basis of the subspace iteration
    double* Qout;    // n x 32 sorted Ritz vectors
    double* X;       // n x 32 G * Qwork
    double* theta;   // 32 Ritz values (descending)
    double* Ca;      // n x n certificate ping
    double* Cb;      // n x n certificate pong
    double* f2;      // 16 squared Frobenius norms of the squaring chain
    int* flags;      // [0] converged [1] need_full [2] svp [3] SI steps [4] certified [5] sweeps of the last SI step
    // large embeddings (n > kEigSmallN): rotated block, projected 32 x 32 problem, Gram of the basis, residuals / norms
    double* Qr; double* Xr; double* Hs; double* Rs; double* Ss; double* res; double* nx;
};
size_t eig_fast_work_doubles(int n);
bool eig_fast_supported(int n);
int eig_fast_max_block(int n);
EigFastWork eig_fast_carve(double* base, int n);
// top1 != 0: "opnorm mode" -- only the dominant eigenpair is wanted and the certificate proves theta_1 = lambda_max.
cudaError_t launch_eig_fast(const double* G, int n, double tau, int nukeA, EigFastWork w, double* lam, double* Vs,
                            double* sigma, double* fvec, int* svp, cudaStream_t st, int64_t* launches, int top1 = 0,
                            int bw = 32, int max_steps = 12);   // bw: block width (16 / 32 columns of Qb); max_steps: subspace steps launched
// Qb = first 32 unit vectors (cold start of the subspace iteration)
cudaError_t launch_init_block(double* Qb, int n, cudaStream_t st, int64_t* launches);
// bounds[0] <= lambda_max(G) <= bounds[1] (device doubles) for a symmetric PSD n x n G by 10 normalised squarings
// (bracket ratio n^(1/2048)).  Ca, Cb: n x n scratch, f2: 16 doubles scratch.
cudaError_t launch_lmax_bounds(const double* G, int n, double* Ca, double* Cb, double* f2, double* bounds,
                               cudaStream_t st, int64_t* launches);
// Qb = Vs[:, 0:32] (skipped on the device when flags != null and flags[1] == 0)
cudaError_t launch_copy_block(const double* Vs, int n, double* Qb, const int* flags, cudaStream_t st,
                              int64_t* launches);

// sigma[i] = sqrt(max(lam[i],0)); svp = #{sigma >= tau}; fvec[i] = nuke ? (sigma-tau)/sigma : 1  (0 beyond svp)
cudaError_t launch_svt_post(const double* lam, int n, double tau, int nukeA, double* sigma, double* fvec,
                            int* svp, cudaStream_t st, int64_t* launches, const int* run_flag = nullptr);

// ----------------------------------------------------------------------------------------------------
// Fused ALM epilogue: one pass over a row tile does  E-step, W, T = W V_r, A = clamp(T diag(f) V_r'),
// Z = D - A - E, Y += mu Z, ||Z||_F^2   (src/robustPCA.jl:188-192, 205-222)
// ----------------------------------------------------------------------------------------------------
struct EpiArgs {
    MatSrc D;
    const double* Ap;   // A_{k-1}
    const double* Yp;   // Y_{k-1}
    double* An;         // A_k      (may alias Ap: the pass is tile-local)
    double* Yn;         // Y_k      (may alias Yp)
    double* Eout;       // optional E_k
    double* Zout;       // optional Z_k = D - A_k - E_k (materialised for the exact stop test)
    double* Wn;         // optional W_{k+1} = D - E_{k+1} + Y_k/mu_{k+1} (materialised SVT input of the next iteration)
    double im_next, eps_next;   // 1/mu_{k+1}, lambda/mu_{k+1}
    double* Uout;       // MODE U only: M x d
    int64_t M, N, ldw;
    const double* Vs;   // N x N sorted right singular vectors (ld N)
    const double* fvec; // N shrink factors (MODE U: 1/sigma)
    const int* svp;     // device scalar: number of columns of Vs to use
    double im, eps, mu;
    int nonnegA, nonnegE;
    double* zz;         // device scalar accumulator for ||Z||_F^2
    // factored low-rank iterate (stream.cu): A_k = clamp(T_k V_k'), T: M x 32 (ld M), V: N x 32 (ld N).  When Tn != null
    // the streaming epilogue reads A_{k-1} from (Tp, Vp, svp_prev) and writes T_k instead of the dense A_k: the dense
    // A is never read or written inside the ALM loop (2 S less HBM traffic per iteration, 2 S less memory).
    const double* Tp;
    const double* Vp;
    int svp_prev;
    double* Tn;
    // hankel=true (:214-216): the tile epilogue only writes the raw reconstruction A' = T diag(f) V_r' into An; the
    // anti-diagonal soft threshold, clamp, Z and Y follow in launch_hankel_finish
    int raw_only;
    // streaming kernels, large N: column range [c0, c1) of one launch (c1 == 0: all columns) and an N x 32 scratch for
    // the GEMM operand V_r diag(f) (set by the solver when N > kEigSmallN)
    int c0, c1;
    double* vf_work;
};
cudaError_t launch_epilogue(const EpiArgs& a, bool hankel, bool mode_u, int sm_count, cudaStream_t st,
                            int64_t* launches);

// Streaming form of the epilogue (stream.cu) for a materialised W and svp <= kStreamMaxRank (svp known on the host):
// T (M x 32 workspace) = W V_r diag(f), then one coalesced element-wise pass.  Needs a.Wn != nullptr.
constexpr int kStreamMaxRank = 32;
// svp_on_device: `svp` is only a GUESS used to pick the rank specialisation; the kernels read the actual rank from the
// device scalar a.svp and return without touching anything when it exceeds stream_rank_pad(svp, a.svp_prev, fact)
// (the caller compares after its next host sync and relaunches).
cudaError_t launch_stream_epilogue(const EpiArgs& a, const double* W, int svp, bool hankel, int sm_count,
                                   cudaStream_t st, int64_t* launches, bool svp_on_device = false);
int stream_rank_pad(int svp, int svp_prev, bool fact);
// TMA-staged form of the same two kernels (stream_tma.cu): 128-row x 8-column boxes through a 4-stage mbarrier ring
bool stream_tma_eligible(const EpiArgs& a, const double* W, int rp, bool hankel);
cudaError_t launch_stream_tma(const EpiArgs& a, const double* W, int rp, int svp, const int* svp_dev, bool hankel,
                              int sm_count, cudaStream_t st);
// can the factored form be used for this (N, svp, svp_prev)?  (two N x RP blocks of V must fit in shared memory)
bool stream_factored_fits(int64_t N, int svp, int svp_prev);
// dense helpers for the factored iterate:  A = clamp(T V')   and   Z = (D - A_k) - E_k  with A_{k-1}, A_k factored
cudaError_t launch_fact_to_dense(const double* T, const double* V, int svp, int64_t M, int64_t N, int nonnegA,
                                 double* A, int sm_count, cudaStream_t st, int64_t* launches);
cudaError_t launch_final_from_factors(const EpiArgs& a, bool hankel, int svp, double* Wout, int sm_count,
                                      cudaStream_t st, int64_t* launches);
// C (M x N, ld M) = X (M x K, ld ldx) * B (K x N, ld K): TMA-free cp.async double-buffered DMMA GEMM (gemm.cu); used for
// the left singular vectors U = W V diag(1/s) of the returned SVD (:238)
cudaError_t launch_gemm_xb(const double* X, int64_t M, int K, int64_t ldx, const double* B, int N, double* C,
                           cudaStream_t st, int64_t* launches);
// same product for any shape / alignment: the DMMA kernel when eligible, else a plain shared-memory-tiled FP64 kernel
cudaError_t launch_gemm_any(const double* X, int64_t M, int K, int64_t ldx, const double* B, int N, double* C,
                            cudaStream_t st, int64_t* launches);
bool gemm_xb_eligible(const double* X, int64_t M, int K, int64_t ldx, int N);
// B[:, c] = V[:, c] * (s_c > 0 ? 1/s_c : 0)
cudaError_t launch_scale_cols_inv(const double* V, const double* sigma, int n, double* B, cudaStream_t st,
                                  int64_t* launches);
cudaError_t launch_z_from_factors(const EpiArgs& a, bool hankel, int svp, double* Z, int sm_count, cudaStream_t st,
                                  int64_t* launches);


// ----------------------------------------------------------------------------------------------------
// Fused one-pass ALM step (fused.cu, n = 256): epilogue of iteration k + Gram of the SVT input of iteration k+1 in ONE
// kernel (thread-block cluster pair per 32-row tile, DSMEM exchange, TMA staging, DMMA Gram).  W is never materialised.
// ----------------------------------------------------------------------------------------------------
constexpr int kFusedN = 256;
constexpr int kFusedMaxRank = 16;
enum FusedGram : int {
    FUSED_GRAM_WNEXT = 0,   // operand = W_{k+1} = (D - E_{k+1}) + Y_k/mu_{k+1}          (the normal step)
    FUSED_GRAM_Z = 1,       // operand = Z_k = (D - A_k) - E_k                            (exact stop test, :225)
    FUSED_GRAM_W = 2,       // operand = W_k from (D, A_{k-1}, Y_{k-1}); nothing written  (first iteration)
    FUSED_GRAM_D = 3        // operand = D                                                (opnorm(D), :177)
};
struct FusedStripTab { uint8_t row[2][8][9]; uint8_t cs[2][8][9]; };
struct FusedArgs {
    MatSrc D;               // dense (TMA) or implicit Hankel signal with lag 1
    const double* Vp;       // V_{k-1}: 256 x >= svp_prev (ld 256)
    const double* Vs;       // V_k:     256 x >= svp      (ld 256)
    const double* fvec;     // shrink factors of iteration k
    int svp, svp_prev;
    double* Yn; int64_t ldy;   // Y_k out (may alias Y_{k-1}: the pass is tile-local)
    double* Tn; int64_t ldt;   // T_k out (compute_T) -- M x 32, ld ldt
    int64_t M;
    double im, eps, mu, im_next, eps_next;
    int nonnegA, nonnegE;
    int compute_T;          // 1: T_k = (W_k V_k) .* f is computed (and written to Tn); 0: T_k is read (Tn_given)
    int write_Y;
    int gram_of;            // FusedGram
    double* partial;        // workspace, fused_partial_doubles(sm_count) doubles
    double* zpart;          // workspace inside partial (set by the launcher)
    const double* VpT;      // packed V_{k-1}' scratch inside partial (set by the launcher)
};
size_t fused_partial_doubles(int sm_count);
FusedStripTab fused_strip_table();      // which 32 x 8 Gram strips every (CTA of the pair, warp) accumulates
bool fused_eligible(const MatSrc& D, bool hankel, int64_t M, int64_t N);
int fused_rank_pad(int svp, int svp_prev);
// G (256 x 256) = Gram of the chosen operand; zz_out (nullable) = ||Z_k||_F^2
cudaError_t launch_alm_fused(const FusedArgs& a, bool hankel, const double* Yp, const double* Tp, const double* Tn_given,
                             double* G, double* zz_out, int sm_count, cudaStream_t st, int64_t* launches);

// element-wise helpers ------------------------------------------------------------------------------
// maxabs: *out = max |D_ij| (out must be zeroed);  init: Y = D / dual, A = 0
cudaError_t launch_maxabs(const MatSrc& D, bool hankel, int64_t M, int64_t N, double* out, int sm_count,
                          cudaStream_t st, int64_t* launches);
// W (optional) = SVT input of the first iteration: (D - E_1) + Y_0/mu_1 with A_0 = 0
cudaError_t launch_init_ya(const MatSrc& D, bool hankel, int64_t M, int64_t N, double dual, double* Y, double* A /*nullable*/,
                           double* W, double im, double eps, int nonnegE, int sm_count, cudaStream_t st,
                           int64_t* launches, int64_t ldy = 0 /* leading dimension of Y; 0 = M */);
// E = soft_th((D - A) + Y/mu, lambda/mu) (+ clamp)
// (E and / or the SVT input Wout = (D - E) + Y/mu; null outputs are skipped)
cudaError_t launch_compute_e(const MatSrc& D, bool hankel, int64_t M, int64_t N, const double* A, const double* Y,
                             double im, double eps, int nonnegE, double* E, int sm_count, cudaStream_t st,
                             int64_t* launches, double* Wout = nullptr);
// out (N x M) = in (M x N)'
cudaError_t launch_transpose(const double* in, int64_t M, int64_t N, double* out, cudaStream_t st,
                             int64_t* launches);

// hankel=true branch of rpca (src/robustPCA.jl:9-21, 214-216, 234-236), single GPU, dense iterate:
//   soft_hankel!(A, eps): every anti-diagonal is soft-thresholded towards its mean  (means from launch_unhankel)
// finish: A = soft_th(A_raw, eps, mean[r+c]); clamp; E from (D, A_prev, Y_prev); Z = D - A - E; Y += mu Z; ||Z||_F^2
cudaError_t launch_hankel_finish(const EpiArgs& a, bool hankel_src, const double* mean, int sm_count, cudaStream_t st,
                                 int64_t* launches);
// dense iterate: A = max(A,0) [nonnegA]; Z = (D - A) - E; Y += mu Z; *zz += ||Z||_F^2   (:217-222; all M x N, ld M)
cudaError_t launch_dense_update(const double* D, double* A, const double* E, double* Y, double* Z, int64_t M, int64_t N,
                                double mu, int nonnegA, double* zz, int sm_count, cudaStream_t st, int64_t* launches);
// X[r,c] = soft_th(X[r,c], eps, mean[r+c]) in place (the final soft_hankel!(E, lambda/mu), :234-236)
cudaError_t launch_soft_hankel_apply(double* X, int64_t M, int64_t N, const double* mean, double eps, int sm_count,
                                     cudaStream_t st, int64_t* launches);

// hankel / unhankel (single channel) ------------------------------------------------------------------
cudaError_t launch_hankel(const double* x, int64_t K, int64_t L, int64_t lag, double* H, cudaStream_t st,
                          int64_t* launches);
cudaError_t launch_unhankel(const double* A, int64_t K, int64_t L, int64_t lag, int64_t Ns, double* y,
                            cudaStream_t st, int64_t* launches);

// multi-channel forms (x: Ns x D column-major, H: K x (L*D) with H[k, l*D + d] = x[k*lag + l, d], :83-90, :53-68)
cudaError_t launch_hankel_mc(const double* x, int64_t Ns, int64_t D, int64_t K, int64_t L, int64_t lag, double* H,
                             cudaStream_t st, int64_t* launches);
cudaError_t launch_unhankel_mc(const double* A, int64_t K, int64_t L, int64_t lag, int64_t Ns, int64_t D, double* y,
                               cudaStream_t st, int64_t* launches);
// A = (H V_sv) V_sv' : the sv > 0 plain-SSA branch of lowrankfilter (:123-125); V = eigenvectors of H'H (ld N)
cudaError_t launch_ssa_project(const MatSrc& H, bool hankel, int64_t M, int64_t N, const double* V, int sv, double* A,
                               int sm_count, cudaStream_t st, int64_t* launches);

// row-sharded unhankel: partial anti-diagonal sums / counts of Hankel rows [r0, r0+Kl) (sum, cnt: Ns doubles, zeroed),
// all-reduced by the caller, then divided
cudaError_t launch_unhankel_partial(const double* A, int64_t r0, int64_t Kl, int64_t L, int64_t lag, int64_t Ns,
                                    double* sum, double* cnt, cudaStream_t st, int64_t* launches);
cudaError_t launch_unhankel_divide(const double* sum, const double* cnt, int64_t Ns, double* y, cudaStream_t st,
                                   int64_t* launches);

// unhankel of the FACTORED iterate A = clamp(T V') (lag 1): sum[k] over the local Hankel rows [r0, r0+Kl); every k in
// [0, Ns) is written (0 where this shard does not contribute); the count is closed-form (divide_count)
cudaError_t launch_unhankel_factors(const double* T, int64_t ldt, const double* V, int svp, int nonnegA, int64_t r0,
                                    int64_t Kl, int64_t n, int64_t Ns, double* sum, int sm_count, cudaStream_t st,
                                    int64_t* launches);
cudaError_t launch_unhankel_divide_count(const double* sum, int64_t K, int64_t n, int64_t Ns, double* y, cudaStream_t st,
                                         int64_t* launches);

// Grassmann averages ----------------------------------------------------------------------------------
enum GaMode : int {
    GA_NORMS = 0,   // t[n] += sum_i X[i,n]^2                                   (src/robustPCA.jl:265)
    GA_DOTS  = 1,   // t[n] += sum_i X[i,n] q[i]                                (:271, and the first :291-293)
    GA_PASS  = 2    // mu_i = (sum_n s[n] X[i,n]) / sumw ; t[n] += sum_i X[i,n] mu_i ; t[N] += sum_i mu_i^2
};                  //                                                          (:291-294, 308-316 in ONE sweep)
// X: d x N (ld), vec: q (GA_DOTS, length d) or mu out (GA_PASS, length d); s: N sign weights; sumw: device scalar
// part (optional, ga_partial_doubles(sm_count) doubles): workspace of the TMA-staged kernel (N <= 256); with it the
// column sums are reduced in fixed order (deterministic), without it the register-prefetch kernel with atomics runs
cudaError_t launch_ga_sweep(GaMode mode, const double* X, int64_t d, int64_t N, int64_t ld, double* vec,
                            const double* s, const double* sumw, double* t, int sm_count, cudaStream_t st,
                            int64_t* launches, double* part = nullptr);
size_t ga_partial_doubles(int sm_count);
// fused tail / head of two components (TMA kernel, same eligibility; cudaErrorNotSupported otherwise): X -= q xs' in
// place (:272); n2[n] += |x_n|^2 of the deflated columns (:265); t2[n] += x_n'q2 when q2 != null (:292)
cudaError_t launch_ga_deflate_fused(double* X, int64_t d, int64_t N, int64_t ld, const double* q, const double* xs,
                                    const double* q2, double* n2, double* t2, double* part, int sm_count,
                                    cudaStream_t st, int64_t* launches);
// xs[n] = t[n] / sqrt(t[N])   (q'x_n from the dot products x_n'mu of the converged iteration, q = mu/|mu|)
cudaError_t launch_ga_xs(const double* t, int64_t N, double* xs, cudaStream_t st, int64_t* launches);
// robust entry-wise averages (:323-333, :349-357): out[j] (length d) from a per-row sort over the N observations;
// kind 1 = trimmed mean (fraction P dropped on each side), 2 = median.  N <= 1024: 8 / 32 rows per tile, one warp per
// row; up to kGaRobustMaxN observations: one CTA per row.  Longer rows take the selection kernels below.
constexpr int kGaRobustMaxN = 16384;
cudaError_t launch_ga_robust(const double* X, int64_t d, int64_t N, int64_t ld, const double* sgn, const double* n2,
                             int kind, double P, double* out, int sm_count, cudaStream_t st, int64_t* launches);
// The same averages for any N (ga_select.cu): per-row radix selection over streaming sweeps of X, same order as
// launch_ga_robust (ascending key, then column; -0.0 == +0.0; NaN keys last).  Keys u = X[j,n] / sqrt(n2[n]) and
// weights w_n = wt[n] sqrt(n2[n]); with n2 == nullptr X holds U itself and wt the weights.  ws: ga_select_bytes().
//   kind 2: out = the median average (:349-357).
//   kind 1: the two boundaries of every row's kept range [floor(P N), floor((1-P) N)) into ws; they depend on X and n2
//           only, so they hold for a whole component.  launch_ga_trimmed_sweep then gives out = the trimmed mean with
//           the current weights (:323-333), summed in a fixed order.
size_t ga_select_bytes(int64_t d, int64_t N, int sm_count);
cudaError_t launch_ga_select(const double* X, int64_t d, int64_t N, int64_t ld, const double* wt, const double* n2,
                             int kind, double P, void* ws, double* out, int sm_count, cudaStream_t st,
                             int64_t* launches);
cudaError_t launch_ga_trimmed_sweep(const double* X, int64_t d, int64_t N, int64_t ld, const double* wt,
                                    const double* n2, double P, const void* ws, double* out, int sm_count,
                                    cudaStream_t st, int64_t* launches);
// s[n] = sign(t[n]) (0 if norms[n]==0), sumw = sum_n s[n]*norms[n]            (:292, :310-312)
cudaError_t launch_ga_signs(const double* t, const double* norms2, int64_t N, double* s, double* sumw,
                            cudaStream_t st, int64_t* launches);
// qnew = mu / sqrt(mm);  dq2 += sum (qnew - qold)^2   (:295-296, 302)   (mm, dq2 device scalars; qnew may alias qold)
cudaError_t launch_ga_update(const double* mu, const double* mm, int64_t d, const double* qold, double* qnew, double* dq2,
                             int sm_count, cudaStream_t st, int64_t* launches);
// ss += sum_i v[i]^2 ;  scale: v *= 1/sqrt(ss)
cudaError_t launch_vec_sumsq(const double* v, int64_t d, double* ss, int sm_count, cudaStream_t st,
                             int64_t* launches);
cudaError_t launch_vec_scale_rsqrt(const double* v, const double* ss, int64_t d, double* out, int sm_count,
                                   cudaStream_t st, int64_t* launches);
// X[i,n] -= q[i] * xs[n]    (:272)
cudaError_t launch_ga_deflate(double* X, int64_t d, int64_t N, int64_t ld, const double* q, const double* xs,
                              int sm_count, cudaStream_t st, int64_t* launches);

}  // namespace tlsq
