/*
 * lpvs.h -- C ABI of liblpvs.so: B200 (sm_100a) least-squares spectral estimation.
 *
 * Drop-in boundary for the hot path of baggepinnen/LPVSpectral.jl.  The reference has no FFI layer of
 * its own; the contract is its exported Julia signatures (src/LPVSpectral.jl:82-97).  Each entry point
 * below names the reference function whose body it replaces.  A thin Julia shim (julia/LPVSpectralB200.jl,
 * see INTEGRATION.md) `ccall`s these; the tests and bench drive the identical ABI through ctypes.
 *
 * Conventions
 *  - every pointer is HOST memory owned by the caller unless the function name ends in `_dev`
 *    (then array arguments are DEVICE pointers on the context's GPU);
 *  - the library never retains a caller pointer after return; every call is synchronous;
 *  - complex outputs are interleaved (re,im) doubles;
 *  - return value: 0 = ok, negative = error code below; message via lpvs_last_error();
 *  - one lpvs_ctx per GPU (one process per GPU); calls on one ctx are serialised internally;
 *  - there is NO CPU fallback: every entry point that computes fails with LPVS_E_CUDA without a GPU.
 */
#ifndef LPVS_H
#define LPVS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lpvs_ctx lpvs_ctx;
typedef struct lpvs_admm lpvs_admm;

enum lpvs_status {
    LPVS_OK = 0,
    LPVS_E_BAD_ARG = -1,     /* reference: ArgumentError / @assert sites (src/lsfft.jl:22, src/windows.jl:31,96, src/lasso.jl:143) */
    LPVS_E_NOT_SPD = -2,     /* Cholesky breakdown; *info = 1-based failing pivot */
    LPVS_E_NONFINITE = -3,   /* NaN/Inf in an input array, or a 0/0 LPV basis normalisation (coulomb with V == 0; the reference returns NaNs) */
    LPVS_E_CUDA = -4,
    LPVS_E_NCCL = -5,        /* reserved: collectives live in the host (torch.distributed / NCCL), not in liblpvs */
    LPVS_E_UNSUPPORTED = -6, /* device older than sm_100; an ADMM problem above 65 536 (padded) unknowns, or the GEMV loop
                                (option LPVS_OPT_ADMM_SYMV at 0) above 25 344 */
    LPVS_E_NOMEM = -7
};

enum lpvs_window_kind { LPVS_WIN_PSD = 0, LPVS_WIN_CSD = 1, LPVS_WIN_COHERE = 2 };
enum lpvs_prox_kind { LPVS_PROX_L1 = 0, LPVS_PROX_L0 = 1, LPVS_PROX_BALL_L0 = 2, LPVS_PROX_GROUP_L2 = 3 };
enum lpvs_phase_mode {
    LPVS_PHASE_AUTO = 0,     /* chain_ref when f is a uniform grid, else direct: always the reference's phase rounding */
    LPVS_PHASE_CHAIN = 1,    /* exact anchors + angle-addition chains with the mathematically EXACT phase 2*pi*f*t: closer to
                                the true basis than the reference, differs from it by up to eps*2*pi*f*t per element */
    LPVS_PHASE_DIRECT = 2,   /* per-element sincos of fl(fl(2*pi*f)*t), the reference's rounding (src/lsfft.jl:34,41) */
    LPVS_PHASE_CHAIN_REF = 3, /* the chains of mode 1, each element turned by fl(fl(2*pi*f)*t) - 2*pi*f*t (5 FP64 ops): the
                                 reference's rounding at chain speed */
    LPVS_PHASE_STRUCTURED = 4, /* uniform grids, opt-in: the Gram matrix from its 3 Nf trigonometric sums (Toeplitz + Hankel in
                                 the frequency index, O(n Nf) instead of O(n Nf^2) work) with the exact phase of the ideal grid
                                 f0 + k df -- the accuracy class of mode 1, not the reference's rounding; everything that is
                                 not a Gram matrix (right-hand sides, operators) runs as in mode 1 */
    LPVS_PHASE_STRUCTURED_REF = 5 /* mode 4 plus the first-order correction of G and b for the reference's phase rounding
                                 eps = fl(fl(2*pi*f)*t) - 2*pi*(f0 + k df)*t: G += D'B + B'D, b += D'y by a half-precision
                                 tensor-core GEMM whose operands are synthesised in registers, eps taken exactly in FP64
                                 (csrc/corr.cu) -- the reference's rounding at 0.38 of mode 3's cost: G agrees with mode 3's
                                 to ~5e-14 max|G| at phases of 2.6e7 rad (the f16 operand rounding of the correction; the
                                 per-element modes agree to 1e-14), which only windows with cond(A'WA) >= 1e8 can tell
                                 apart; opt-in; everything that is not a Gram matrix runs as in mode 3 */
};
enum lpvs_option {
    LPVS_OPT_PHASE_MODE = 0,   /* lpvs_phase_mode */
    LPVS_OPT_WINDOW_BATCH = 1, /* windows factorised per batch (bounds workspace), default auto */
    LPVS_OPT_JITTER = 2,       /* 1 (default): unweighted ls_spectral / ls_spectral_lpv are solved to the accuracy of the
                                  reference's SVD / pivoted QR of [A; lambda I] (refinement on the operator, shifted CholeskyQR
                                  when needed: rank-deficient defaults work, *info = LPVS_INFO_QR); weighted / windowed solves
                                  re-factor a numerically singular problem with ridge max(lambda, Nreg*eps*max diag G)
                                  (*info = LPVS_INFO_JITTER).  0: plain Cholesky everywhere, LPVS_E_NOT_SPD on breakdown */
    LPVS_OPT_ADMM_CHECK_EVERY = 3, /* residual test cadence inside the device loop; 1 (default) = every iteration (Q12) */
    LPVS_OPT_SHARD_EXCHANGE = 6,   /* one ADMM problem over several GPUs, exchange per iteration (set identically on every rank):
                                      2 (default) all-reduce of the partial products by peer stores, prox computed redundantly on
                                        every rank: ONE cross-GPU step and two grid barriers per iteration;
                                      1 reduce-scatter + all-gather with per-CTA arrival counters (two steps, one barrier);
                                      0 reduce-scatter + all-gather with flags raised by CTA 0 (two steps, three barriers) */
    LPVS_OPT_ADMM_M32 = 7,         /* 1: ADMM problems created while set store the inverse (G + I/mu)^-1 in single precision and
                                      accumulate in double -- half the bytes per iteration; what the Float32 instantiation of
                                      ls_sparse_spectral[_lpv] (src/lasso.jl:85, eltype-generic) uses.  Single GPU, SYMV loop.
                                      0 (default): double */
    LPVS_OPT_TRSV_FLOW = 5,        /* triangular solves of ONE large problem: 1 (default) flag-chained dataflow kernel,
                                      0 the grid-barrier kernel (one barrier per 128-block step) */
    LPVS_OPT_ADMM_SYMV = 4         /* x-update kernel: -1 auto (default), 0 GEMV over the full symmetric inverse (8 Np^2 B/iter,
                                      Np <= 25 344), 1 SYMV over its lower triangle (4 Np^2 B/iter) */
};

/* info flags returned by solvers */
#define LPVS_INFO_JITTER 1 /* a WEIGHTED (Gram / LU in the reference) problem was numerically singular: jitter ridge used */
#define LPVS_INFO_DUAL 3   /* informational: Nreg >= N, solved in the sample space: x = A'(A A' + lambda^2 I)^-1 y */
#define LPVS_INFO_QR 2     /* informational: the unweighted / LPV solve took the shifted-CholeskyQR path (ill-conditioned A) */

int lpvs_version(void);
int lpvs_device_count(void);
int lpvs_init(int device, lpvs_ctx** ctx);
void lpvs_destroy(lpvs_ctx* ctx); /* also frees ADMM handles of this context that were not freed; they become invalid */
const char* lpvs_last_error(const lpvs_ctx* ctx);
int lpvs_set_option(lpvs_ctx* ctx, int key, double value);
/* enqueue all work of this context on the caller's CUDA stream (cudaStream_t as void*; NULL = the context's own
 * stream).  Lets a host framework order the library's kernels with its own work and time them with its events. */
int lpvs_set_stream(lpvs_ctx* ctx, void* stream);
/* cumulative number of kernels this context launched (bench.py's gpu_launches) */
int64_t lpvs_launch_count(const lpvs_ctx* ctx);
/* device time [ms] and launch count of the Gram kernel(s) during the last API call (bench.py's roofline) */
int lpvs_last_gram_timing(const lpvs_ctx* ctx, double* ms, int64_t* launches, double* flops);
/* device time [ms] between the first and last operation the last compute call enqueued on the context's stream
 * (H2D/D2H copies of the host-pointer entry points included) */
int lpvs_last_call_ms(const lpvs_ctx* ctx, double* ms);
/* cudaMalloc/cudaFree/cudaMemcpy wrappers so a host language without CUDA bindings can keep inputs resident */
int lpvs_dev_alloc(lpvs_ctx* ctx, int64_t bytes, void** dptr);
int lpvs_dev_free(lpvs_ctx* ctx, void* dptr);
int lpvs_dev_upload(lpvs_ctx* ctx, void* dptr, const void* hptr, int64_t bytes);
int lpvs_dev_download(lpvs_ctx* ctx, void* hptr, const void* dptr, int64_t bytes);
int lpvs_sync(lpvs_ctx* ctx);
/* the context's device workspaces are grow-only (a cfg5b-sized call leaves ~17 GB of tables behind): give them back.  ADMM
 * handles keep their own memory and stay valid. */
int lpvs_release_workspace(lpvs_ctx* ctx);

/* ---- window bookkeeping: DSP.arraysplit semantics used by Windows2/Windows3 (src/windows.jl:27-36,94-104) ---- */
/* K = N >= n ? (N-n) div (n-noverlap) + 1 : 0 ; noverlap < 0 means n>>1 */
int64_t lpvs_window_count(int64_t N, int n, int noverlap);

/* ---- get_fourier_regressor + Gram (src/lsfft.jl:26-49, :77) -- parity/bench entry ----
 * G (Nreg x Nreg, full symmetric, reference column order: cos block then -sin block) = A' diag(W) A,
 * b (Nreg) = A' diag(W) y.  W and y may be NULL (W=1, b not produced). Nreg = 2Nf - (f[0]==0). */
int lpvs_gram_fourier(lpvs_ctx* ctx, const double* y, const double* t, int64_t N, const double* f, int Nf,
                      const double* W, double* G, double* b);

/* ---- ls_spectral(y,t,f; lambda) and ls_spectral(y,t,f,W; lambda)  (src/lsfft.jl:62-80) ----
 * W == NULL: x = argmin |Ax-y|^2 + lambda^2 |x|^2, to the accuracy of svd([A; lambda I]) \ [y; 0]
 *            (fourier_solve, src/utilities.jl:56-60); the default call with Nreg = N+1 > N is fine
 * W != NULL: x = (A'WA + lambda I)^-1 A'Wy  (src/lsfft.jl:77)
 * x: Nf complex (fourier2complex, src/utilities.jl:62-73). */
int lpvs_ls_spectral(lpvs_ctx* ctx, const double* y, const double* t, int64_t N, const double* f, int Nf,
                     const double* W, double lambda, double* x, int* info);

/* ---- ls_spectral of C channels sampled at the same t (no reference equivalent) ----
 * Column c of X is what lpvs_ls_spectral(Y + c*ldY, t, N, f, Nf, W, lambda) computes, to the same accuracy; the Gram matrix,
 * its factors and (for the unweighted solve) the QR objects depend only on t, W and f and are built once for all channels.
 * Y: C channels of N samples, channel c at Y + c*ldY; ldY >= N, C >= 1.  X: Nf x C complex, column-major (channel c at
 * X + 2*c*Nf doubles, fourier2complex order).  info (may be NULL): C ints, the route flag lpvs_ls_spectral reports for that
 * channel (0, LPVS_INFO_DUAL, LPVS_INFO_QR or LPVS_INFO_JITTER); with LPVS_E_NOT_SPD (the factor is shared) every entry holds
 * the pivot.  LPVS_E_NONFINITE names the first channel holding a NaN or Inf.  A channel's column and info are independent,
 * bit for bit, of the other channels of the call (which, how many, in what order).  The host form uploads each channel with
 * its own copy (no pitch limit on ldY); the _dev form takes Y, t and W (nullable) on the device, f, X and info on the host. */
int lpvs_ls_spectral_multi(lpvs_ctx* ctx, const double* Y, int C, int64_t ldY, const double* t, int64_t N,
                           const double* f, int Nf, const double* W, double lambda, double* X, int* info);
int lpvs_ls_spectral_multi_dev(lpvs_ctx* ctx, const double* d_Y, int C, int64_t ldY, const double* d_t, int64_t N,
                               const double* f, int Nf, const double* d_W, double lambda, double* X, int* info);

/* ---- Base.merge(yf, w::Windows2), the re-assembly step of mapwindows (src/windows.jl:50-70; SURVEY 8f n4) ----
 * pieces: K x n doubles (window k = samples [k (n-noverlap), +n), as lpvs_window_count counts them), out: N doubles =
 * the overlap-average: covering windows added in window order, divided by max(count, 1) (uncovered tail samples stay 0). */
int lpvs_merge_windows(lpvs_ctx* ctx, const double* pieces, int64_t K, int n, int noverlap, int64_t N, double* out);

/* ---- tls_spectral(y,t,f) (src/lsfft.jl:87-99; SURVEY 8f n3) ----
 * Total least squares: x = -V[1:n, n+1] / V[n+1, n+1], V the right singular vectors of [A y].  Computed as the eigenvector of
 * the smallest eigenvalue of [A y]'[A y] (the Gram pass gives A'A and A'y) by inverse iteration on the factorised bordered
 * matrix; *iters (may be NULL) = inverse-iteration steps taken.  The reference's default f is default_freqs(t)[1:end-1]. */
int lpvs_tls_spectral(lpvs_ctx* ctx, const double* y, const double* t, int64_t N, const double* f, int Nf, double* x,
                      int* iters);

/* ---- ls_windowpsd / ls_windowcsd / ls_cohere (src/lsfft.jl:112-126, 140-156, 176-193) ----
 * One weighted ls_spectral per window (window weights W[n], shared), reduced on device.
 * `sums` holds the raw cross-window sums for windows [k_begin,k_end) (multi-GPU: ranks take disjoint ranges and
 * add their sums before finalising):
 *   PSD:    Nf   doubles  sum |x|^2
 *   CSD:    2Nf  doubles  [Re sum xy conj(xu) | Im ...]
 *   COHERE: 4Nf  doubles  [Syy | Suu | Re Syu | Im Syu]
 * lpvs_ls_window_finalize applies /K^2 (PSD), /K (CSD) or |Syu|^2/(Suu Syy) (COHERE) with Julia's abs2 order.
 * LPVS_E_NOT_SPD names the absolute index of the failing window in both forms.  The sums do not depend on
 * LPVS_OPT_WINDOW_BATCH; in LPVS_PHASE_STRUCTURED_REF a window's last bits depend on the call's window range [k_begin, k_end)
 * (the correction is scaled by max |t| over it), so ranks of a sharded run differ from one GPU in the last bits. */
int lpvs_ls_window_sums(lpvs_ctx* ctx, int kind, const double* y, const double* u, const double* t, int64_t N,
                        const double* f, int Nf, const double* W, int n, int noverlap, double lambda,
                        int64_t k_begin, int64_t k_end, double* sums, int* info);
int lpvs_ls_window_sums_dev(lpvs_ctx* ctx, int kind, const double* d_y, const double* d_u, const double* d_t,
                            int64_t N, const double* f, int Nf, const double* W, int n, int noverlap,
                            double lambda, int64_t k_begin, int64_t k_end, double* sums, int* info);
int lpvs_ls_window_finalize(int kind, const double* sums, int Nf, int64_t K, double* out);
/* all windows on this GPU + finalize; out: PSD Nf reals, CSD Nf complex, COHERE Nf reals; *K = window count */
int lpvs_ls_window(lpvs_ctx* ctx, int kind, const double* y, const double* u, const double* t, int64_t N,
                   const double* f, int Nf, const double* W, int n, int noverlap, double lambda, double* out,
                   int64_t* K, int* info);

/* ---- cross-spectral / coherence MATRICES of C channels sampled at the same t (no reference equivalent) ----
 * The windowed estimators above for every pair of channels at once.  Per window the Gram matrix A'WA and its Cholesky factor
 * depend only on t, W and f, so they are built ONCE and the C right-hand sides A'W Y[:, c] are solved against that factor.
 * Y: C channels of N samples, channel c at Y + c*ldY (a column-major N x C matrix has ldY = N); ldY >= N, C >= 1.
 * sums: Nf*C*C complex (interleaved), [f][i][j] = sum over windows [k_begin, k_end) of x_i(f) conj(x_j(f)), the raw sum
 * lpvs_ls_window_sums(LPVS_WIN_CSD, y = Y[:,i], u = Y[:,j]) accumulates.  S is exactly Hermitian (S_ji = conj(S_ij)) and
 * independent of LPVS_OPT_WINDOW_BATCH bit for bit (in LPVS_PHASE_STRUCTURED_REF the last bits depend on the call's window
 * range, as in lpvs_ls_window_sums).  *info as lpvs_ls_window_sums (LPVS_INFO_JITTER, or the pivot with LPVS_E_NOT_SPD and the
 * absolute window index in the message).  The host form uploads only the samples of [k_begin, k_end); the _dev form takes Y and t on the device.
 * Ranks of a multi-GPU run take disjoint window ranges and add their sums before finalising. */
int lpvs_ls_window_matrix_sums(lpvs_ctx* ctx, const double* Y, int C, int64_t ldY, const double* t, int64_t N,
                               const double* f, int Nf, const double* W, int n, int noverlap, double lambda,
                               int64_t k_begin, int64_t k_end, double* sums, int* info);
int lpvs_ls_window_matrix_sums_dev(lpvs_ctx* ctx, const double* d_Y, int C, int64_t ldY, const double* d_t, int64_t N,
                                   const double* f, int Nf, const double* W, int n, int noverlap, double lambda,
                                   int64_t k_begin, int64_t k_end, double* sums, int* info);
/* no context needed; K = total window count (0 gives NaN, as lpvs_ls_window_finalize):
 *   LPVS_WIN_PSD:    out Nf*C reals [f][c]        = S_cc / K^2
 *   LPVS_WIN_CSD:    out Nf*C*C complex [f][i][j] = S_ij / K
 *   LPVS_WIN_COHERE: out Nf*C*C reals [f][i][j]   = abs2(S_ij) / (S_jj S_ii), Julia's abs2 order (the diagonal is exactly 1) */
int lpvs_ls_window_matrix_finalize(int kind, const double* sums, int Nf, int C, int64_t K, double* out);

/* ---- windowed estimators with estimator = ls_sparse_spectral (src/lsfft.jl:121,150-151,184-185 -> the weighted
 * method src/lasso.jl:105-126; exercised by test/test_lasso.jl:36) ----
 * Every window is an independent ADMM problem on Quadratic(A'WA, A'Wy) (sign quirk Q13 kept), x0 = 0 (init=false),
 * run on the device to its own stop test ||x-z||_2 < tol (or `iters`); sums as lpvs_ls_window_sums, to be finished with
 * lpvs_ls_window_finalize.  iters_done / residuals (may be NULL): one entry per window and channel,
 * [(k_end-k_begin)][nrhs], nrhs = 1 (PSD) or 2 -- what the reference prints when a window stops (src/lasso.jl:164). */
int lpvs_ls_window_sparse_sums(lpvs_ctx* ctx, int kind, const double* y, const double* u, const double* t, int64_t N,
                               const double* f, int Nf, const double* W, int n, int noverlap, int prox_kind,
                               double prox_param, double mu, int64_t iters, double tol, int64_t k_begin,
                               int64_t k_end, double* sums, int64_t* iters_done, double* residuals, int* info);

/* ---- sparse cross-spectral / coherence MATRICES of C channels sampled at the same t (no reference equivalent) ----
 * lpvs_ls_window_sparse_sums for every pair of channels at once.  Per window the inverse M = (A'WA + I/mu)^-1 is built ONCE,
 * each channel's ADMM problem (right-hand side A'W Y[:, c]) runs ONCE against it to its own stop test, and
 * S_ij = sum over windows of z_i conj(z_j) is accumulated on the device.  Y, C, ldY, the window range and sums as
 * lpvs_ls_window_matrix_sums (sums Nf*C*C complex [f][i][j], finished with lpvs_ls_window_matrix_finalize); prox_kind,
 * prox_param, mu, iters and tol as lpvs_ls_window_sparse_sums (L1, L0, IndBallL0; mu in (0, 1]).  iters_done / residuals
 * (may be NULL): [(k_end-k_begin)][C].  A channel's z, iteration count and residual are bitwise independent of the other
 * channels of the call (which, how many, in which order) and of LPVS_OPT_WINDOW_BATCH, so S is exactly Hermitian and the
 * coherence diagonal is exactly 1 wherever S_ii != 0.  In LPVS_PHASE_STRUCTURED_REF the last bits depend on the call's
 * window range, as in lpvs_ls_window_matrix_sums.  LPVS_E_NOT_SPD names the absolute window in both forms.  The host form
 * uploads only the samples of [k_begin, k_end) and checks them for NaN/Inf; the _dev form takes Y and t on the device. */
int lpvs_ls_window_matrix_sparse_sums(lpvs_ctx* ctx, const double* Y, int C, int64_t ldY, const double* t, int64_t N,
                                      const double* f, int Nf, const double* W, int n, int noverlap, int prox_kind,
                                      double prox_param, double mu, int64_t iters, double tol, int64_t k_begin,
                                      int64_t k_end, double* sums, int64_t* iters_done, double* residuals, int* info);
int lpvs_ls_window_matrix_sparse_sums_dev(lpvs_ctx* ctx, const double* d_Y, int C, int64_t ldY, const double* d_t,
                                          int64_t N, const double* f, int Nf, const double* W, int n, int noverlap,
                                          int prox_kind, double prox_param, double mu, int64_t iters, double tol,
                                          int64_t k_begin, int64_t k_end, double* sums, int64_t* iters_done,
                                          double* residuals, int* info);

/* ---- ls_spectral_lpv (src/lsfft.jl:239-259; basis src/utilities.jl:23-36, src/lsfft.jl:195-207) ----
 * params: Nf*Nvv complex (Nvv = coulomb ? 2Nv : Nv), column order f + k*Nf.
 * Sigma (may be NULL): (2 Nf Nvv)^2 doubles = var(e) * inv(Ar'Ar + lambda I).  fva: fraction of variance explained. */
int lpvs_ls_spectral_lpv(lpvs_ctx* ctx, const double* Y, const double* X, const double* V, int64_t N,
                         const double* w, int Nf, int Nv, double lambda, int coulomb, int normalize,
                         double* params, double* Sigma, double* fva, int* info);

/* ---- ls_windowpsd_lpv (src/lsfft.jl:267-277; Windows3, src/windows.jl:94-104) ----
 * Rect windows of n samples overlapping by `noverlap` (< 0 means n>>1): window k is the sample range
 * [k (n-noverlap), +n) of Y, X, V (uploaded once), estimated by ls_spectral_lpv on the window's OWN basis centres.
 * S: Nf doubles = sum over windows of |sum_k x[f,k]|^2 (not normalised, as the reference).  fva (may be NULL): one
 * fraction of variance explained per window (the reference warns per window when it is < 0.9); size it with
 * lpvs_window_count(N, n, noverlap).  *K = number of windows. */
int lpvs_ls_windowpsd_lpv(lpvs_ctx* ctx, const double* Y, const double* X, const double* V, int64_t N,
                          const double* w, int Nf, int Nv, int n, int noverlap, double lambda, int coulomb,
                          int normalize, double* S, double* fva, int64_t* K, int* info);

/* ---- ls_spectral_lpv / ls_windowpsd_lpv of C output channels sharing X, V and w ----
 * Channel c is at Y + c*ldY (ldY >= N).  The basis tables, the Gram matrix, its factors and (on the QR route) the QR
 * objects depend only on X, V and w, so they are built once for all channels.  Column c, info[c], fva[c] and var_e[c]
 * are what the single-channel call returns for Y + c*ldY, to the same accuracy, and bitwise independent of the other
 * channels of the call.  LPVS_E_NONFINITE names the first channel holding a NaN or Inf; with LPVS_E_NOT_SPD every info
 * entry holds the shared pivot.
 * lpvs_ls_spectral_lpv_multi: params Nf*Nvv*C complex, channel c at params + 2*c*Nf*Nvv doubles (ls_spectral_lpv's
 * column order).  Sigma0 (may be NULL): (2 Nf Nvv)^2 doubles = inv(Ar'Ar + lambda I), the same for every channel; the
 * Sigma of channel c is var_e[c] * Sigma0.  var_e, fva (may be NULL): C doubles, var(e_c) (n - 1) and the fraction of
 * variance explained.  info (may be NULL): C ints, the route flag lpvs_ls_spectral_lpv reports for that channel.
 * lpvs_ls_windowpsd_lpv_multi: S is Nf x C, channel c at S + c*Nf, each column the raw sum of lpvs_ls_windowpsd_lpv.
 * fva (may be NULL): [K][C].  info (may be NULL): C ints, each the OR of the channel's flags over its windows; the
 * message of LPVS_E_NOT_SPD names the window. */
int lpvs_ls_spectral_lpv_multi(lpvs_ctx* ctx, const double* Y, int C, int64_t ldY, const double* X, const double* V,
                               int64_t N, const double* w, int Nf, int Nv, double lambda, int coulomb, int normalize,
                               double* params, double* Sigma0, double* var_e, double* fva, int* info);
int lpvs_ls_windowpsd_lpv_multi(lpvs_ctx* ctx, const double* Y, int C, int64_t ldY, const double* X, const double* V,
                                int64_t N, const double* w, int Nf, int Nv, int n, int noverlap, double lambda, int coulomb,
                                int normalize, double* S, double* fva, int64_t* K, int* info);

/* ---- ADMM (src/lasso.jl:136-171) behind ls_sparse_spectral / ls_sparse_spectral_lpv (src/lasso.jl:27-126) ----
 * create: builds the Gram on device, factorises (G + I/mu), keeps everything resident.
 *   W == NULL  -> LeastSquares(A,y):   x-update solves (G + I/mu) x = A'y + (z-u)/mu
 *   W != NULL  -> Quadratic(A'WA,A'Wy): x-update solves (Q + I/mu) x = (z-u)/mu - q   (sign quirk Q13 kept)
 *   x0 (Nreg, reference order) may be NULL (zeros).  init != 0: x0 = ridge LS with ridge lambda_init^2 (Q14).
 * run: up to max_iters more iterations on device without host sync; stops when ||x-z||_2 < tol.
 * Size: up to 65 536 padded unknowns (Np, the unknowns rounded up to 128), else LPVS_E_UNSUPPORTED; the bound comes from
 * the index and launch arithmetic, the largest size run is Np = 46 464.  Create needs G and the inverse workspace at
 * once, 16 Np^2 bytes (39 GB at Np = 49 152); without that much free device memory -- checked after the ridge start of
 * init != 0, whose workspaces the context keeps -- it returns LPVS_E_NOMEM before the Gram is built.  The GEMV loop keeps
 * the whole rhs in shared memory and stops at Np = 25 344 on a 148-SM B200; the SYMV loop (auto above that) keeps only
 * the 128-blocks each CTA touches and runs every size.
 * The shim loops run(printerval) to reproduce the reference's prints / callback (SURVEY H6). */
int lpvs_admm_create_fourier(lpvs_ctx* ctx, const double* y, const double* t, int64_t N, const double* f, int Nf,
                             const double* W, int prox_kind, double prox_param, double mu, const double* x0,
                             int init, double lambda_init, lpvs_admm** h);
int lpvs_admm_create_lpv(lpvs_ctx* ctx, const double* y, const double* X, const double* V, int64_t N,
                         const double* w, int Nf, int Nv, int coulomb, int normalize, double lambda, double mu,
                         lpvs_admm** h);
int lpvs_admm_run(lpvs_admm* h, int64_t max_iters, double tol, int64_t* iters_done, double* residual,
                  int* converged);
/* ---- ONE problem sharded over the GPUs of a node (SURVEY 8e, third row): one process per GPU, every rank creates the
 * SAME problem, then
 *   lpvs_admm_shard_begin(h, rank, world)   re-plans the loop for this rank's share of the inverse and allocates the
 *                                           exchange region;
 *   lpvs_admm_shard_handle(h, buf64)        exports the region (CUDA IPC, 64 bytes) -- the host all-gathers these;
 *   lpvs_admm_shard_connect(h, handles)     maps the peers' regions (world x 64 bytes, rank order).
 * After a host barrier, lpvs_admm_run (same max_iters / tol on every rank) iterates with device-initiated peer stores
 * over NVLink (LPVS_OPT_SHARD_EXCHANGE, default: one all-reduce of the partial products per iteration, prox computed
 * redundantly on every rank), no host or NCCL call inside the loop.  NormL1 / NormL0, and with the default exchange
 * IndBallL0 and the group prox of lpvs_admm_create_lpv.  lpvs_admm_get / _result are valid on every rank after a host barrier that follows
 * the run. */
int lpvs_admm_shard_begin(lpvs_admm* h, int rank, int world);
int lpvs_admm_shard_handle(lpvs_admm* h, void* handle64);
int lpvs_admm_shard_connect(lpvs_admm* h, const void* handles);
int lpvs_admm_size(const lpvs_admm* h); /* length of x / z in reference order */
int lpvs_admm_get(lpvs_admm* h, double* x, double* z);
/* fourier2complex(z) (Nf complex) or LPV params (Nf*Nv complex, un-permuted as src/lasso.jl:67-68) */
int lpvs_admm_result(lpvs_admm* h, double* out);
/* device time [ms] of the last lpvs_admm_run loop kernel and its algorithmic bytes per iteration */
int lpvs_admm_last_timing(const lpvs_admm* h, double* ms, double* bytes_per_iter);
void lpvs_admm_free(lpvs_admm* h);

/* ---- parity entry: z = prox_{gamma g}(v) computed by the ADMM loop's own device routines (the g-update of
 * src/lasso.jl:153: ProximalOperators prox!(z, proxg, x+u, mu)).  v, z: Nreg = 2Nf - (zero_first != 0) doubles in the
 * reference's order [cos block; sin block].  NormL1 / NormL0 / IndBallL0; ties of IndBallL0 go to the lower REFERENCE index. */
int lpvs_prox_fourier(lpvs_ctx* ctx, int prox_kind, double prox_param, double gamma, const double* v, int Nf,
                      int zero_first, double* z);

/* one-shot conveniences mirroring the Julia functions */
int lpvs_ls_sparse_spectral(lpvs_ctx* ctx, const double* y, const double* t, int64_t N, const double* f, int Nf,
                            const double* W, int prox_kind, double prox_param, double mu, int init,
                            double lambda_init, int64_t iters, double tol, double* x, int64_t* iters_done,
                            double* residual);
int lpvs_ls_sparse_spectral_lpv(lpvs_ctx* ctx, const double* y, const double* X, const double* V, int64_t N,
                                const double* w, int Nf, int Nv, int coulomb, int normalize, double lambda,
                                double mu, int64_t iters, double tol, double* params, int64_t* iters_done,
                                double* residual);

/* ---- row-sharded Gram for very tall problems (SURVEY 8e): partial packed Gram on DEVICE so the host can
 * all-reduce it (NCCL via torch.distributed / ncclAllReduce) before lpvs_solve_packed_dev ----
 * d_packed: Np*Np + 2*Np doubles (internal tiled layout, lower tiles + 2 rhs), see lpvs_packed_size. */
int64_t lpvs_packed_size(int Nf);
int lpvs_gram_partial_dev(lpvs_ctx* ctx, const double* d_y, const double* d_u, const double* d_t,
                          const double* d_W, int64_t N, const double* f, int Nf, double* d_packed);
/* x: nrhs * Nf complex; ridge is added as given (caller picks lambda or lambda^2) */
int lpvs_solve_packed_dev(lpvs_ctx* ctx, double* d_packed, const double* f, int Nf, int nrhs, double ridge,
                          double* x, int* info);

#ifdef __cplusplus
}
#endif
#endif /* LPVS_H */
