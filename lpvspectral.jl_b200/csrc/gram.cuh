// Gram formation with on-the-fly basis synthesis: G = A' diag(W) A, b = A' diag(W) [y u].
// A is never materialised in HBM: each CTA synthesises its [128 functions] x [32 samples] basis tiles in
// shared memory and feeds them to FP64 DMMA.  Replaces get_fourier_regressor + A'Wd*A (src/lsfft.jl:26-49,77),
// the LPV row loop (src/lsfft.jl:244-248) and the LeastSquares constructor's A'A (src/lasso.jl:51,98).
#pragma once
#include "common.cuh"

namespace lpvs {

// GRAM_CHAIN: exact-phase anchors + angle-addition chains.  GRAM_CHAINREF: the same chains, each element then turned by the
// tiny angle fl(fl(2 pi f) t) - 2 pi f t, so the basis carries the REFERENCE's phase rounding (src/lsfft.jl:34,41) -- 5 FP64
// ops per element instead of a sincos.  GRAM_DIRECT: per-element sincos of the reference-rounded phase (any grid).
enum GramMode { GRAM_CHAIN = 0, GRAM_DIRECT = 1, GRAM_LPV = 2, GRAM_CHAINREF = 3 };
__host__ __device__ constexpr bool gram_is_chain(int mode) { return mode == GRAM_CHAIN || mode == GRAM_CHAINREF; }

// Internal column layout (size Np = 128*nblk): block q holds "complex columns" cc = 64q .. 64q+63;
// internal index p = 128q + (cc%64) for the real part (cos, or Re A for LPV) and 128q + 64 + (cc%64) for the
// second part (-sin, or Im A).  Fourier: cc = frequency index.  LPV: cc = f + k*Nf (reference order).
// Columns with cc >= ncc, and the -sin column of a zero frequency, are identically zero ("dummy"): the
// factorisation gives them a unit diagonal so they decouple.
struct GramArgs {
    const double* t;  // sample positions, absolute index
    const double* y;  // rhs 0 (nullable)
    const double* u;  // rhs 1 (nullable)
    const double* W;  // weights (nullable = 1)
    int w_abs;        // 0: W indexed by in-problem sample index (shared window weights); 1: by absolute index
    long long start0; // problem p covers absolute samples [start0 + p*hop, start0 + p*hop + n)
    long long hop;
    int n;
    long long s_end;  // samples >= s_end are invalid (ragged last split)
    int ncc;  // valid complex columns (Nf, or Nf*Nvv for LPV)
    int nblk; // Np / 128
    int nrhs;
    int fuse_rhs;  // set by launch_gram: b for nrhs == 1 is accumulated inside the diagonal tiles
    // GRAM_CHAIN tables, indexed [row * tbl_ns + (s - tbl_base)]: anc rows [0, nblk) block anchors, [nblk, nblk + GRP)
    // group powers (launch_anchor_table)
    const double2* anc;
    const double2* del;
    long long tbl_base;
    long long tbl_ns;
    // GRAM_CHAINREF: per complex column (w, dw): w = fl(2 pi f), dw = w - 2 pi (f_block + fl(8 g df) + j df) (double-double, host)
    const double2* wtab;
    // GRAM_DIRECT
    const double* f;
    // GRAM_LPV tables: E[fi * tbl_ns + s'], Kt[ki * tbl_ns + s']
    const double2* E;
    const double* Kt;
    int lpv_nf;
    // output
    double gscale, bscale;
    double* G;  // per problem Np x Np row-major: lower 128x128 tiles; of a diagonal tile only the 16x32 pieces that touch
                // the lower triangle are written -- entries above the diagonal are unspecified, no consumer reads them
    long long strideG;
    double* B;  // per problem [2][Np]
    long long strideB;
};

size_t gram_smem_bytes();
// grid = (nblk*(nblk+1)/2, nproblems); returns the number of kernels launched
int launch_gram(int mode, const GramArgs& a, int nproblems, cudaStream_t st);

// only b = A' diag(W) [y u] (grid = (nblk, nproblems)); the adjoint of the synthesised operator
int launch_gram_rhs(int mode, const GramArgs& a, int nproblems, cudaStream_t st);

// B[p][c][Np] = A' diag(W) Y[:, c] for C channels sampled at a.t: channel c starts at Y + c ldY and is indexed like a.t;
// a.B / a.strideB hold C x Np doubles per problem (a.y, a.u, a.nrhs unused).  GRAM_CHAIN, GRAM_CHAINREF, GRAM_DIRECT or GRAM_LPV;
// grid = (nblk, nproblems, C / RHS_MC rounded up)
constexpr int RHS_MC = 4;  // channels per CTA
int launch_gram_rhs_multi(int mode, const GramArgs& a, const double* Y, long long ldY, int C, int nproblems,
                          cudaStream_t st);

// Chain anchor tables, exact phase (double-double turns): anc has nblk + GRP rows of ns entries -- rows [0, nblk) the first
// frequency of every 64-frequency block, rows [nblk, nblk + GRP) the turn by anchor_group_step(j, df) from there to chain
// group j -- and del the per-sample step rotation e^{-i 2 pi df t}.  (Round 1 kept one anchor per 8 frequencies: 8 nblk rows,
// 2.1 GB at BASELINE cfg2; this layout is 0.8 GB and costs one complex multiply per 8 synthesised elements.)
constexpr int anchor_rows(int nblk) { return nblk + GRP; }
inline double anchor_group_step(int j, double df) { return (double)(GRP * j) * df; }  // the double the device phase uses
void launch_anchor_table(const double* t, long long s0, long long ns, const double* f, int nblk, double df, double2* anc,
                         double2* del, cudaStream_t st);
// LPV factor tables: E[fi][s] = (cos, -sin)(w_fi * X_s) (reference rounding), Kt[ki][s] = RBF activations
void launch_lpv_tables(const double* X, const double* V, long long N, const double* w, int Nf, int Nvv,
                       const double* centers, double gamma, int coulomb, int normalize, double2* E, double* Kt,
                       int* nonfinite /* device flag, bit 2 set on a 0/0 normalisation; nullable */, cudaStream_t st);

// ---- LPVS_PHASE_STRUCTURED (structured.cu): Gram matrix and right-hand sides of a uniform-grid Fourier basis from
// trigonometric sums.  Per problem the sums live in one array of 64-blocks: [0, nzg) the blocks for G (Z-, Z+; one family when
// f0 = 0), then nby blocks per right-hand side; the table has one row per block, then GRP group powers, then the step.
struct StructuredLayout {
    bool alias;         // f0 == 0: Z- is the head of Z+
    int zm_off, zp_off; // offsets (in sums) of Z-(0) and Z+(0)
    int zy_off[2];      // offsets of Zy(0), Zu(0)
    int nzg, nby, nzb;  // blocks for G, blocks per right-hand side, all blocks
    int nrows;          // table rows: nzb + GRP + 1
};
StructuredLayout structured_layout(double f0, int Nf, int nrhs);
void structured_row_freqs(double f0, double df, int Nf, int nrhs, double* out /* 2 * nrows doubles: (hi, lo) per row */);
struct SumArgs {
    const double* t;
    const double* W;  // nullable = 1
    const double* y;  // right-hand sides (weights W y, W u of the last 2 * nby blocks); nullable with nby = 0
    const double* u;
    int w_abs;        // as GramArgs
    long long start0, hop;
    int n;
    long long s_end;
    const double2* tab;  // [row][tbl_ns]
    long long tbl_base, tbl_ns;
    int nzg, nby, nzb;
    double2* Z;          // per problem nzb * 64 sums
    long long strideZ;
};
struct FillArgs {
    const double2* Z;
    long long strideZ;
    int zm_off, zp_off, zy_off[2];
    int ncc, nblk, zero_first;
    double gscale;
    double* G;  // per problem Np x Np, every lower 128-tile written in full
    long long strideG;
};
// frow_dev holds the rows of the nrhs = 2 layout; the table gets the first nzb block rows + the GRP + 1 trailing rows
void launch_sum_tables(const double* t, long long s0, long long ns, const double2* frow_dev, int nzb, int nzb_full,
                       double2* tab, cudaStream_t st);
int launch_trig_sums(const SumArgs& a, int nproblems, cudaStream_t st);
void launch_sum_parts(double2* out, const double2* parts, int count, long long stride, int nparts, int accumulate,
                      cudaStream_t st);
int launch_gram_fill(const FillArgs& a, int nproblems, cudaStream_t st);
void launch_rhs_from_sums(const FillArgs& a, int nrhs, double bscale, double* B, long long strideB, int nproblems,
                          cudaStream_t st);

// ---- LPVS_PHASE_STRUCTURED_REF (corr.cu): first-order correction of the structured Gram matrix / right-hand sides for the
// reference's phase rounding, G += D'B + B'D, b += D'[y u], by a half-precision tensor-core GEMM over per-sample tables
struct CorrArgs {
    const double* t;
    const double* W;  // nullable = 1
    const double* y;  // right-hand sides (launch_rhs_corr only)
    const double* u;
    int w_abs;        // as GramArgs
    long long start0, hop;
    int n;
    long long s_end;
    int ncc, nblk, nrhs;
    const double2* wtab;  // per complex column (fl(2 pi f_k), fl(2 pi f_k) - 2 pi (f0 + k df)), zero beyond ncc
    double wmax, dwmax;   // max |w|, max |dw| over the columns
    double df;
    // tables of the sample range [tbl_base, tbl_base + tbl_ns) (launch_corr_tables), rows of tbl_ns entries
    long long tbl_base, tbl_ns;
    // sample range whose max |t| sets the scales: [scal_base, scal_base + scal_ns), the table range when scal_ns == 0
    long long scal_base, scal_ns;
    double* scal;   // [2]: max |t| (of the scale range), max |W| -> the power-of-two scales
    uint4* eps;     // [8 nblk][tbl_ns]: eps S 2^-7 of the 8 columns of a chain group, f16
    float2* anc;    // [8 nblk][tbl_ns]: (cos, -sin) of the reference phase of the group's first column
    float2* step;   // [tbl_ns]: (cos, -sin)(2 pi df t)
    float* wf;      // float(W wsc): by in-problem sample index (w_abs = 0) or by table index (w_abs = 1)
    double gscale, bscale;
    double* G;  // per problem Np x Np, lower 128-tiles (read-modify-write, every tile in full)
    long long strideG;
    double* B;  // per problem [2][Np] (read-modify-write)
    long long strideB;
};
size_t corr_table_bytes_per_sample(int nblk);
// fills a.scal, a.eps, a.anc, a.step for the table range and a.wf from W[w0 .. w0 + nw); returns the number of kernels launched
int launch_corr_tables(const CorrArgs& a, long long w0, long long nw, cudaStream_t st);
int launch_gram_corr(const CorrArgs& a, int nproblems, cudaStream_t st);  // returns the number of kernels launched
int launch_rhs_corr(const CorrArgs& a, int nproblems, cudaStream_t st);
void structured_ref_wtab(double f0, double df, const double* f, int Nf, int ncol, double* out /* 2 ncol */, double* wmax,
                         double* dwmax);

}  // namespace lpvs
