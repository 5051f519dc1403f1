// Internal context / workspace definitions for liblpvs.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/lpvs.h"
#include "chol.cuh"
#include "gram.cuh"

namespace lpvs {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

enum BufSlot {
    BUF_T = 0, BUF_Y, BUF_U, BUF_W, BUF_F, BUF_ANC, BUF_DEL, BUF_G, BUF_B, BUF_LINV, BUF_INFO, BUF_PART, BUF_SUMS,
    BUF_X, BUF_MISC, BUF_YINV, BUF_E, BUF_K, BUF_V, BUF_CENT, BUF_LSQ_R, BUF_LSQ_V, BUF_LSQ_Y, BUF_LSQ_LI, BUF_LSQ_A,
    BUF_LSQ_BT, BUF_LSQ_G2, BUF_WTAB, BUF_FLAGS, BUF_PSD, BUF_TRSM, BUF_WIN_ITS, BUF_WIN_RES, BUF_SFREQ, BUF_SANC, BUF_ZSUM, BUF_ZPART, BUF_CWTAB, BUF_CPART, BUF_CSCAL, BUF_CEPS, BUF_CANC, BUF_CSTEP, BUF_CWF,
    BUF_MC_PART, BUF_MC_ACT, BUF_MC_NRM, BUF_MC_G, BUF_MC_W, BUF_MC_X, BUF_MC_X2, BUF_COUNT
};

}  // namespace lpvs

struct lpvs_ctx {
    int device = 0;
    int sms = 148;
    cudaStream_t st = nullptr;      // stream in use
    cudaStream_t own_st = nullptr;  // the context's own stream
    lpvs::Lookahead la{};           // aux stream + events of the look-ahead factorisation (single large problems)
    std::string err;
    std::recursive_mutex mu;  // serialises every call on this context; recursive so composite entry points hold it throughout
    int phase_mode = LPVS_PHASE_AUTO;
    int window_batch = 0;
    int jitter = 1;
    int admm_check_every = 1;
    int admm_symv = -1;  // -1 auto, 0 GEMV over full M, 1 SYMV over the lower triangle
    int admm_m32 = 0;    // ADMM handles created while set keep the inverse in single precision (Float32 callers)
    int trsv_flow = 1;   // single-problem triangular solves: dataflow kernel (1) or grid-barrier kernel (0)
    int shard_exchange = 2;  // sharded ADMM exchange: 0 flag hops (3 barriers, 2 exchanges), 1 arrival counters, 2 all-reduce by
                             // peer stores + redundant prox (2 barriers, 1 exchange per iteration)
    lpvs::DevBuf buf[lpvs::BUF_COUNT];
    int64_t launches = 0;
    // Gram kernel timing of the last API call
    std::vector<cudaEvent_t> ev;
    int ev_used = 0;
    double gram_ms = 0.0;
    int64_t gram_launches = 0;
    double gram_flops = 0.0;
    cudaEvent_t ev_call0 = nullptr, ev_call1 = nullptr;
    int call_depth = 0;
    int* d_nonfinite = nullptr;  // set by the upload-time scan of host inputs
    std::vector<double> wtab_host;      // staging of the GRAM_CHAINREF phase table (kept alive across the async upload)
    std::vector<double> sfreq_host;     // staging of the LPVS_PHASE_STRUCTURED row frequencies
    std::vector<double> cwtab_host;     // staging of the LPVS_PHASE_STRUCTURED_REF (w, dw) table
    std::vector<lpvs_admm*> live_admm;  // handles created on this context and not yet freed
};

namespace lpvs {

using Lock = std::lock_guard<std::recursive_mutex>;

int fail(lpvs_ctx* c, int code, const char* fmt, ...);

// brackets a public compute call with events on the context stream (outermost call only)
struct CallTimer {
    lpvs_ctx* c;
    explicit CallTimer(lpvs_ctx* ctx) : c(ctx) {
        if (c && c->call_depth++ == 0) {
            cudaEventRecord(c->ev_call0, c->st);
            if (c->d_nonfinite) cudaMemsetAsync(c->d_nonfinite, 0, sizeof(int), c->st);
        }
    }
    ~CallTimer() {
        if (c && --c->call_depth == 0) cudaEventRecord(c->ev_call1, c->st);
    }
};

#define LPVS_CU(ctx, call)                                                                      \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess)                                                                  \
            return lpvs::fail(ctx, LPVS_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                              __FILE__, __LINE__);                                              \
    } while (0)

// grow-only workspace
void* ws_raw(lpvs_ctx* c, int slot, size_t bytes);
template <class T>
inline T* ws(lpvs_ctx* c, int slot, size_t count) {
    return reinterpret_cast<T*>(ws_raw(c, slot, count * sizeof(T)));
}

// description of a Fourier basis on the internal tiled layout
struct FourierPlan {
    int Nf = 0, Nreg = 0, nblk = 0, Np = 0, ngroups = 0;
    int zero_first = 0;
    int mode = GRAM_CHAIN;
    double f0 = 0.0, df = 0.0, dd = 1.0;
    const double* d_f = nullptr;
    const double2* d_wtab = nullptr;  // GRAM_CHAINREF: (fl(2 pi f), fl(2 pi f) - 2 pi (f_anchor + j df)) per complex column
    bool structured = false;          // LPVS_PHASE_STRUCTURED: Gram matrices from trigonometric sums (structured.cu); mode = GRAM_CHAIN
    const double2* d_sfreq = nullptr; // ... double-double frequencies of the sum-table rows
    bool structured_ref = false;      // LPVS_PHASE_STRUCTURED_REF: + first-order correction for the reference's phase (corr.cu); mode = GRAM_CHAINREF
    const double2* d_cwtab = nullptr; // ... (fl(2 pi f_k), fl(2 pi f_k) - 2 pi (f0 + k df)) per complex column
    double cw_max = 0.0, cdw_max = 0.0;
};
int make_fourier_plan(lpvs_ctx* c, const double* f, int Nf, FourierPlan* plan);
inline int pcol(int k) { return (k >> 6) * 128 + (k & 63); }

void gram_timer_begin(lpvs_ctx* c);
void gram_timer_end(lpvs_ctx* c, double flops, int launches);
void gram_timer_reset(lpvs_ctx* c);
int gram_timer_resolve(lpvs_ctx* c);

// G (Np x Np lower tiles) and B ([2][Np]) for ONE problem over samples [0,N) of device arrays; split over samples
// when the tile count alone cannot fill the GPU.  d_W indexed by absolute sample (nullable).
int gram_single(lpvs_ctx* c, const FourierPlan& pl, const double* d_t, const double* d_y, const double* d_u,
                const double* d_W, int64_t N, int nrhs, double* d_G, double* d_B);

// factor + solve one problem in place: d_G -> L, d_B -> x (internal layout); returns pivot info in *info_host
// d_ridge (device, one value per problem) replaces `ridge` when given
// robust (ONE problem): TRSM tiles refined once (CholArgs::trsm_scratch), full forward + backward solve afterwards
int factor_solve(lpvs_ctx* c, int ncc, int zero_first, int Np, double* d_G, double* d_B, int nrhs, double ridge,
                 int nproblems, int* info_host /* nproblems or null */, const double* d_maxdiag = nullptr,
                 double tol_scale = 0.0, const double* d_ridge = nullptr, bool robust = false);

// The regressor as an operator, synthesised on the fly with the REFERENCE's rounding (lsq.cu): Fourier
// fl(fl(cos(fl(fl(2 pi f) t))) dd) (src/lsfft.jl:34-44) or the LPV tables (src/lsfft.jl:244-248).
struct OpArgs {
    int mode = GRAM_DIRECT;  // GRAM_DIRECT (Fourier) or GRAM_LPV
    const double* t = nullptr;
    const double* f = nullptr;
    double dd = 1.0;
    const double2* E = nullptr;
    const double* Kt = nullptr;
    long long tbl_ns = 0;
    int lpv_nf = 1;
    int ncc = 0;  // valid complex columns
    int zero_first = 0;
    long long N = 0;
};
// tls_spectral on device: in d_G = A'A (lower tiles, destroyed), d_B[0] = A'y; out d_B[0] = x (internal layout)
int tls_solve(lpvs_ctx* c, int Np, int ncc, int zero_first, const double* d_y, long long N, double* d_G, double* d_B,
              int* iters_out);
// x = argmin |A x - y|^2 + lam^2 |x|^2 to the accuracy of a QR / SVD of [A; lam I] (see lsq.cu).  In: d_G = Gram matrix of
// ANY phase mode (lower tiles, destroyed), d_B[0] = A'y; out: d_B[0] = x (internal layout).  regram() must rebuild d_G / d_B
// (only called if the shifted factorisation itself breaks down).  *info: 0, or LPVS_INFO_QR when the QR path ran.
int ls_solve_accurate(lpvs_ctx* c, const OpArgs& op, int Np, int zero_first, const double* d_y, double* d_G, double* d_B,
                      double lam, const std::function<int()>& regram, int* info);

// ---- ls_spectral of C channels at shared sample times (lsq.cu) ----
// out[c][i] = sum_k op(M)[i][k] V[c][k], op(M) = trans ? M' : M (row-major, ld); tri 0 full, 1 lower, 2 upper (tiles of op(M)
// outside that triangle must be zero and are skipped).  Channels with d_active[c] == 0 are not written (d_active nullable).
int skinny_apply(lpvs_ctx* c, const double* M, long long ld, bool trans, int tri, int rows, long long K, const double* V,
                 long long ldv, int C, const int* d_active, double* out, long long ldo);
// d_X = L^-1 (n x n, zeros above the diagonal) from a factor d_L and its kept diagonal-block inverses; d_S: n x n scratch
int factor_inverse(lpvs_ctx* c, const double* d_L, const double* d_diag_inv, int n, double* d_X, double* d_S);
// d_out[c] = (L L')^-1 d_B[c] = X' (X d_B[c]) for C vectors of length n (ld n); d_tmp: C x n; in place allowed
int llt_solve_multi(lpvs_ctx* c, const double* d_X, int n, const double* d_B, int C, const int* d_active, double* d_out,
                    double* d_tmp);
// d_out[c] = A' diag(W) R[c] ([C][Np]) through k_gram_rhs_multi over sample splits; base: the basis fields of a GramArgs
// (t, W, w_abs, ncc, nblk, tables, f, bscale) with start0 = 0, s_end = N
int adjoint_apply_multi(lpvs_ctx* c, const GramArgs& base, int mode, int Np, const double* d_R, long long ldr, int C,
                        double* d_out);
// d_X[c] = (L L')^-1 A' diag(W) Y[c] ([C][Np]) for C channels Y[c] = d_Y + c ldY, L the factor factor_solve left in d_L
// (its diagonal-block inverses in BUF_LINV); base, mode: the adjoint's basis, as adjoint_apply_multi
int chol_solve_multi(lpvs_ctx* c, const GramArgs& base, int mode, int Np, const double* d_L, const double* d_Y,
                     long long ldY, int C, double* d_X);
// ls_solve_accurate for C channels Y[c] = d_Y + c ldY: d_G = A'A (destroyed; regram() rebuilds it), out d_X [C][Np]
// (internal layout), info[c] = 0 / LPVS_INFO_DUAL / LPVS_INFO_QR / LPVS_INFO_JITTER, the route the channel took
int ls_solve_accurate_multi(lpvs_ctx* c, const OpArgs& op, int Np, int zero_first, const double* d_Y, long long ldY, int C,
                            double* d_G, double lam, const std::function<int()>& regram, double* d_X, int* info);
// R[c] = Y[c] - A X[c] for C channels (X: [C][Np] internal layout, R: ld ldr >= op.N), through k_op_apply_multi
void op_residual_multi(lpvs_ctx* c, const OpArgs& op, const double* d_X, int Np, const double* d_Y, long long ldY,
                       double* d_R, long long ldr, int C);

// device scratch for the flag-chained TRSV (null = use the grid-barrier kernel)
inline int* trsv_flags(lpvs_ctx* c, int nb) { return c->trsv_flow ? ws<int>(c, BUF_FLAGS, (size_t)2 * nb) : nullptr; }

// shared helpers (api.cu)
// reads the upload-time non-finite flag (synchronises the stream); LPVS_E_NONFINITE if any host input had NaN/Inf
int inputs_finite(lpvs_ctx* c);
int upload(lpvs_ctx* c, int slot, const double* h, int64_t n, double** d);
// samples [s0, s0 + ns) of C host channels (channel c at Y + c ldY) to BUF_Y, channel c at *d_Y + c ns
int upload_channels(lpvs_ctx* c, const double* Y, int C, int64_t ldY, int64_t s0, int64_t ns, double** d_Y);
// out[0] <- min(out[0], c) over the channels c (blockIdx.y) of Y holding a NaN / Inf
__global__ void k_first_nonfinite_channel(const double* __restrict__ Y, long long ldY, long long N, int* out);
void fill_basis_args(const FourierPlan& pl, GramArgs& g);
// ridge LS on device arrays; on return *d_x points at the internal-layout solution ([nrhs][Np], BUF_B)
int ls_solve_dev(lpvs_ctx* c, const FourierPlan& pl, const double* d_t, const double* d_y, const double* d_u,
                 const double* d_W, int64_t N, int nrhs, double ridge, bool allow_jitter, double** d_x, int* info);
// out[i] (+)= sum_p parts[p*stride + i]
void reduce_parts(lpvs_ctx* c, double* out, const double* parts, long long count, long long stride, int nparts,
                  int accumulate);
void launch_gather_ref(lpvs_ctx* c, const double* G, const double* B, int Np, int half, int zero_first, int nref,
                       double* Gout, double* bout);
void launch_x_to_complex(lpvs_ctx* c, const double* X, int Np, int ncx, int zero_first, int nrhs, double* out);
void launch_scatter_ref_vec(lpvs_ctx* c, const double* xin, int half, int zero_first, int nref, int Np, double* xout);

// LPV basis (lpv.cu)
struct LpvPlan {
    int Nf = 0, Nv = 0, Nvv = 0, ncc = 0, nblk = 0, Np = 0;
    int coulomb = 0, normalize = 1;
    int64_t N = 0;
    const double2* d_E = nullptr;
    const double* d_K = nullptr;
};
int lpv_prepare(lpvs_ctx* c, const double* X, const double* V, int64_t N, const double* w, int Nf, int Nv,
                int coulomb, int normalize, LpvPlan* pl);
// G (Np x Np lower tiles), B[0] = Ar'y for one LPV problem
int lpv_gram(lpvs_ctx* c, const LpvPlan& pl, const double* d_y, double* d_G, double* d_B);

// ADMM plumbing (admm.cu)
lpvs_admm* admm_new(lpvs_ctx* c);
void admm_release_all(lpvs_ctx* c);  // lpvs_destroy: free handles the caller leaked
void admm_delete(lpvs_admm* h);
void admm_set_problem(lpvs_admm* h, int kind, int Np, int ncc, int zero_first, int nref, int half, int prox,
                      double pparam, double mu, int quad, int lpv_nf, int lpv_nvv);
int admm_set_groups(lpvs_ctx* c, lpvs_admm* h, const std::vector<int>& goff, const std::vector<int>& gmem);
int admm_check_size(lpvs_ctx* c, long long Np);
int admm_check_memory(lpvs_ctx* c, long long Np);
int admm_finish_create(lpvs_ctx* c, lpvs_admm* h, double* d_G, const double* d_q, const double* d_x0);
// one CTA per window: d_M [nw] Np x Np inverses, d_B [nw][2][Np] rhs in / z out; d_iters, d_res: [nw][nrhs]
int admm_batch_run(lpvs_ctx* c, const double* d_M, double* d_B, int Np, int nrhs, int nw, int prox, double pparam,
                   double mu, int quad, long long iters, double tol, long long* d_iters, double* d_res, int ref_half,
                   int zero_first);
// one CTA per (window, chunk of channels): d_B [nw][C][Np] rhs in / z out; d_iters, d_res: [nw][C]
int admm_multi_run(lpvs_ctx* c, const double* d_M, double* d_B, int Np, int C, int nw, int prox, double pparam,
                   double mu, long long iters, double tol, long long* d_iters, double* d_res, int ref_half,
                   int zero_first);

}  // namespace lpvs
