// Blocked FP64 Cholesky / triangular solves / SPD inverse on the internal tiled layout (Np = 128*nb, row-major,
// lower triangle).  Replaces the reference's dense solves: svd([A;lam I])\ (src/utilities.jl:58), the N-rhs LU
// (src/lsfft.jl:77), pivoted QR (src/utilities.jl:52), inv(AA'AA+lam I) (src/lsfft.jl:254) and the CG x-update
// (src/lasso.jl:151), all on the Gram matrix.
#pragma once
#include "common.cuh"

namespace lpvs {

enum GemmMode {
    GM_TRSM = 0,       // A_ik <- A_ik * Linv_kk'                       (i > k)
    GM_SYRK_RIGHT = 1, // A_ij -= A_ik A_jk'                            (i >= j > k)
    GM_SYRK_LEFT = 2,  // A_ik -= sum_{j<k} A_ij A_kj'                  (i >= k)
    GM_TRTRI_A = 3,    // Y_ki  = Y[k, k:i) * L[i, k:i)'                (k < i)
    GM_TRTRI_B = 4,    // Y_ki <- -Y_ki * Linv_ii'
    GM_LAUUM = 5,      // M_ab  = Y[a, a:nb) * Y[b, a:nb)'              (a >= b), M written into G
    GM_SYRK_COL = 6,   // GM_SYRK_RIGHT restricted to block column k+1  (the next panel: look-ahead)
    GM_SYRK_REST = 7,  // GM_SYRK_RIGHT for block columns >= k+2
    GM_TRSM_RES = 8,   // S_i <- S_i - A_ik L_kk'   (S = copy of the pre-TRSM tile: the residual of the inverse-based TRSM)
    GM_TRSM_FIX = 9    // A_ik <- A_ik + S_i Linv_kk'   (one step of iterative refinement of the TRSM)
};

// Look-ahead for ONE large problem (right-looking): the trailing update of columns >= k+2 runs on `aux` while the next
// diagonal block is factorised on the main stream.  Null = plain in-order factorisation.
struct Lookahead {
    cudaStream_t aux;
    cudaEvent_t e_trsm, e_rest;
};

struct CholArgs {
    double* G;  // per problem Np x Np row-major (lower)
    long long strideG;
    double* Y;  // inverse-transpose workspace (upper), same shape
    long long strideY;
    double* Linv;  // per problem nb blocks of 128x128 (ld 128)
    long long strideLinv;
    int* info;  // per problem: 0 ok, else 1-based failing pivot (internal index)
    // optional numerical-rank test: a pivot <= maxdiag[prob] * tol_scale counts as breakdown (null = only <= 0)
    const double* maxdiag;
    double tol_scale;
    int Np, nb;
    // optional (ONE problem): nb x 128 x 128 doubles.  When set, every TRSM tile A_ik Linv_kk' is refined once against L_kk
    // (A_ik += (A_ik0 - A_ik L_kk') Linv_kk').  Applying a diagonal block through its explicit inverse loses cond(L_kk) eps;
    // on matrices with many tiny pivots (rank-deficient Gram matrices with a 1e-13 shift) that is enough to drive later
    // pivots negative -- a substitution-based TRSM (LAPACK) or this one refinement step does not (tools, DESIGN 1a).
    double* trsm_scratch;
    // optional right-hand sides [nrhs][Np] per problem: the forward substitution L y = b rides along with the
    // factorisation (k_potf2 finishes y_k = Linv_kk r_k, the TRSM tiles apply r_i -= L_ik y_k), b is overwritten by y
    double* rhs;
    long long strideRhs;
    int nrhs;
};

size_t potf2_smem_bytes();
size_t gemm_smem_bytes();

// diagonal: G[i][i] = dummy(i) ? 1 : G[i][i] + ridge[prob or 0]
void launch_diag_prepare(double* G, long long strideG, int Np, int ncc, int zero_first, const double* ridge_dev,
                         double ridge, int nproblems, cudaStream_t st);
void launch_potf2(const CholArgs& a, int k, int nproblems, cudaStream_t st);
void launch_gemm(int mode, const CholArgs& a, int k, int ntiles, int nproblems, cudaStream_t st);
// Y_kk = Linv_kk' for all k
void launch_init_y(const CholArgs& a, int nproblems, cudaStream_t st);
// mirror lower tiles of G into the upper triangle
void launch_symmetrize(double* G, long long strideG, int Np, int nproblems, cudaStream_t st);
// B[p][r][Np] <- (L L')^{-1} B, nrhs <= 2, one CTA per problem
// fwd_done: B already holds y = L^-1 b (fused forward substitution), only L' x = y remains
// flow_flags (2*nb ints of device scratch, nullable): enables the flag-chained single-problem kernel
void launch_trsv(const CholArgs& a, double* B, long long strideB, int nrhs, int nproblems, cudaStream_t st,
                 bool fwd_done = false, int* flow_flags = nullptr);
// after potrf: B[p][c][Np] <- (L L')^{-1} B for C right-hand sides per problem (k_trsm_multi, DMMA panels of
// trsm_multi_chunk(C) channels, one CTA per problem and chunk); problems with a.info != 0 are left untouched
void launch_trsm_multi(const CholArgs& a, double* B, long long strideB, int C, int nproblems, cudaStream_t st);
int trsm_multi_chunk(int C);
// max_i G[i][i] over non-dummy i  -> out[prob]
void launch_max_diag(const double* G, long long strideG, int Np, int ncc, int zero_first, double* out,
                     int nproblems, cudaStream_t st);

// full factorisation driver (left-looking when batched, right-looking for few large problems); returns launches
int potrf(const CholArgs& a, int nproblems, int sms, cudaStream_t st, const Lookahead* la = nullptr);
// after potrf: Y = L^-T (upper 128-tiles of a.Y; tiles below the diagonal are not written). returns launches
int trtri(const CholArgs& a, int nproblems, cudaStream_t st);
// after potrf: M = (L L')^{-1} written (full symmetric) into G; uses Y. returns launches
int potri(const CholArgs& a, int nproblems, cudaStream_t st);

__host__ __device__ inline bool is_dummy_col(int p, int ncc, int zero_first) {
    int q = p >> 7, r = p & 127;
    int part = r >> 6;
    int cc = q * 64 + (r & 63);
    if (cc >= ncc) return true;
    return zero_first && part == 1 && cc == 0;
}

}  // namespace lpvs
