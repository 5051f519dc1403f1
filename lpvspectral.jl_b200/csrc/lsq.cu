// Least squares on the regressor itself, for the estimators the reference does NOT solve through a Gram matrix:
// unweighted ls_spectral -> fourier_solve = svd([A; lam I]) \ [y; 0]        (src/utilities.jl:56-60)
// ls_spectral_lpv        -> real_complex_bs = [Ar; lam I] \ [Y; 0], pivoted QR (src/utilities.jl:49-54)
// Those results are defined by A to cond([A; lam I])*eps; a Cholesky of A'A + lam^2 I is only good to cond^2*eps and breaks
// down on the reference's own defaults (default_freqs gives Nreg = N+1; lam = 1e-10 / 1e-8).  The tensor-core work is
// kept -- the Gram matrix and its Cholesky factor become a PRECONDITIONER -- and the accuracy comes from the operator:
//
//   1. G~ = A'A (fused synthesis + DMMA, any phase mode), L L' = G~ + max(lam^2, n eps max diag G~) I   (one factorisation)
//   2. corrected semi-normal equations with the REFERENCE-ROUNDED operator synthesised on the fly:
//        r = y - A x,  dx = (L L')^-1 (A' r - lam^2 x),  x += dx
//      converges in 1-4 steps when cond(A)^2 * eps is small against the shift (every well-conditioned problem);
//   3. otherwise (rank deficient / cond(A) >~ 1e5): shifted CholeskyQR.  Q1 = [A; lam I] L^-T has condition ~1e4 however
//      bad A is, so the Gram matrix of the MATERIALISED Q1 can be factorised safely:
//        Y = L^-T (TRTRI), Q1' = L^-1 [A' | lam I] (one triangular DMMA GEMM), G2 = Q1'Q1 (DMMA SYRK), G2 z = Q1'[y;0],
//        x = Y z.
//      Forward error ~ cond([A; lam I]) * eps, the class of the reference's SVD / QR (measured against numpy's gesdd, geqrf
//      and gelsy, which differ among themselves by as much: tests/test_gpu_rankdef.py, DESIGN.md section 1).
#include <math.h>
#include <stdio.h>

#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "ctx.h"

namespace lpvs {

namespace {

constexpr double EPS = 2.220446049250313e-16;

// element (s, cc) of the reference-rounded regressor: (Re, Im) part pair of complex column cc
__device__ __forceinline__ double2 op_elem(const OpArgs& a, int cc, long long s, double ts) {
    if (a.mode == GRAM_DIRECT) {
        const double2 v = cis_reference(a.f[cc], ts);
        return make_double2(__dmul_rn(v.x, a.dd), __dmul_rn(v.y, a.dd));  // fl(fl(cos) * dd), src/lsfft.jl:42-44
    }
    const int fi = cc % a.lpv_nf, ki = cc / a.lpv_nf;
    const double2 e = a.E[(long long)fi * a.tbl_ns + s];
    const double k = a.Kt[(long long)ki * a.tbl_ns + s];
    return make_double2(__dmul_rn(e.x, k), __dmul_rn(e.y, k));
}

// out[s] = (y ? y[s] : 0) - sum_cc Re A[s,cc] x[p(cc)] + Im A[s,cc] x[p(cc)+64]; lane = sample, warp = column slice
__global__ void __launch_bounds__(256) k_op_apply(const __grid_constant__ OpArgs a, const double* __restrict__ x,
                                                  const double* __restrict__ y, double* __restrict__ out) {
    __shared__ double part[8][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long long s = (long long)blockIdx.x * 32 + lane;
    const bool valid = s < a.N;
    const long long sc = valid ? s : a.N - 1;
    const double ts = a.mode == GRAM_DIRECT ? a.t[sc] : 0.0;
    double acc = 0.0;
    for (int cc = w; cc < a.ncc; cc += 8) {
        const double2 v = op_elem(a, cc, sc, ts);
        const int p = (cc >> 6) * 128 + (cc & 63);
        acc = fma(v.x, x[p], acc);
        acc = fma(v.y, x[p + 64], acc);
    }
    part[w][lane] = acc;
    __syncthreads();
    if (w == 0 && valid) {
        double t = 0.0;
#pragma unroll
        for (int q = 0; q < 8; q++) t += part[q][lane];
        out[s] = (y ? y[s] : 0.0) - t;
    }
}

// Arow[s][p] = A[s, p] in the internal column layout, rows [0, Nr) (rows >= N and dummy columns are zero)
__global__ void __launch_bounds__(256) k_materialize(const __grid_constant__ OpArgs a, double* __restrict__ Arow, int Np,
                                                     long long Nr) {
    const int j = threadIdx.x & 63, q = blockIdx.y, cc = q * 64 + j;
    const long long s = (long long)blockIdx.x * 4 + (threadIdx.x >> 6);
    if (s >= Nr) return;
    double2 v = make_double2(0.0, 0.0);
    if (s < a.N && cc < a.ncc) v = op_elem(a, cc, s, a.mode == GRAM_DIRECT ? a.t[s] : 0.0);
    if (a.zero_first && cc == 0) v.y = 0.0;
    Arow[s * Np + q * 128 + j] = v.x;
    Arow[s * Np + q * 128 + 64 + j] = v.y;
}

// Y = X' (upper) and the ridge block of Q1': Bt[i][Nr + k] = scale(k) X[i][k], scale = lam for real columns, 1 for dummy
// columns (their unit diagonal keeps G2 non-singular).  X is lower triangular with explicit zeros above the diagonal.
__global__ void __launch_bounds__(256) k_transpose_linv(const double* __restrict__ X, int Np, int ncc, int zero_first,
                                                        double lam, double* __restrict__ Y, double* __restrict__ Bt,
                                                        long long ldbt, long long Nr) {
    __shared__ double tile[32][33];
    const int bi = blockIdx.y, bk = blockIdx.x;  // input rows 32*bi.., columns 32*bk..
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int i = bi * 32 + r, k = bk * 32 + tx;
        const double v = X[(long long)i * Np + k];
        tile[r][tx] = v;
        Bt[(long long)i * ldbt + Nr + k] = v * (is_dummy_col(k, ncc, zero_first) ? 1.0 : lam);
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) Y[(long long)(bk * 32 + r) * Np + bi * 32 + tx] = tile[tx][r];
}

// B operand stored [K][N] (N contiguous): a [KC x 128] slab into a [KC][LDN] smem tile; LDN == 4 (mod 16) keeps the DMMA
// fragment loads (k = lane & 3, n = lane >> 2) conflict-free per half warp
constexpr int LDN = TB + 4;
static_assert(KC * LDN <= TILE_D, "the [k][n] tile must fit the [n][k] tile's slot");
__device__ __forceinline__ void load_tile_async_kn(double* dst, const double* src, long long ld, int tid) {
#pragma unroll
    for (int i = 0; i < (TB * KC / 2) / NTHREADS; i++) {
        const int q = tid + i * NTHREADS;
        const int row = q >> 6, seg = q & 63;
        cp_async16(dst + row * LDN + 2 * seg, src + (long long)row * ld + 2 * seg);
    }
}
__device__ __forceinline__ void mma_step_kn(const double* __restrict__ pa, const double* __restrict__ pb, int kk,
                                            double (&acc)[4][8][2]) {
    double a[4], b[8];
#pragma unroll
    for (int i = 0; i < 4; i++) a[i] = pa[i * 8 * LDT + 4 * kk];
#pragma unroll
    for (int j = 0; j < 8; j++) b[j] = pb[4 * kk * LDN + 8 * j];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
}

// acc += A[128 x (k0..k1)] * op(B): BKN ? B[(k0..k1) x 128] (row-major, ldb) : B[128 x (k0..k1)]' -- 3-stage cp.async ring,
// one __syncthreads per chunk.  A / B point at column / row k0 already.
constexpr int NT_STAGES = 3;
template <bool BKN>
__device__ __forceinline__ void gemm_mainloop(const double* A, long long lda, const double* B, long long ldb, int nchunks,
                                              double* sm, double (&acc)[4][8][2]) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int wm = w & 3, wn = w >> 2;
    auto load = [&](int stage, int chunk) {
        double* dst = sm + stage * 2 * TILE_D;
        load_tile_async(dst, A + (long long)chunk * KC, lda, tid);
        if (BKN)
            load_tile_async_kn(dst + TILE_D, B + (long long)chunk * KC * ldb, ldb, tid);
        else
            load_tile_async(dst + TILE_D, B + (long long)chunk * KC, ldb, tid);
    };
#pragma unroll
    for (int p = 0; p < NT_STAGES - 1; p++) {
        if (p < nchunks) load(p, p);
        cp_async_commit();
    }
    const int fragA = (32 * wm + (lane >> 2)) * LDT + (lane & 3);
    const int fragB = BKN ? (lane & 3) * LDN + 64 * wn + (lane >> 2) : (64 * wn + (lane >> 2)) * LDT + (lane & 3);
    int st_cur = 0;
    for (int c = 0; c < nchunks; c++) {
        cp_async_wait<NT_STAGES - 2>();  // chunk c has landed (only the newest group may still be in flight)
        __syncthreads();                 // ... for every thread, and everyone has left the stage refilled below
        const int st_fill = st_cur == 0 ? NT_STAGES - 1 : st_cur - 1;
        if (c + NT_STAGES - 1 < nchunks) load(st_fill, c + NT_STAGES - 1);
        cp_async_commit();
        const double* pa = sm + st_cur * 2 * TILE_D + fragA;
        const double* pb = sm + st_cur * 2 * TILE_D + TILE_D + fragB;
#pragma unroll
        for (int kk = 0; kk < KC / 4; kk++) {
            if (BKN)
                mma_step_kn(pa, pb, kk, acc);
            else
                mma_step(pa, pb, kk, acc);
        }
        st_cur = st_cur == NT_STAGES - 1 ? 0 : st_cur + 1;
    }
    cp_async_wait<0>();
}

__device__ __forceinline__ void store_tile(double* C, long long ldc, double alpha, const double (&acc)[4][8][2]) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int wm = w & 3, wn = w >> 2;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int row = 32 * wm + 8 * i + (lane >> 2);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const int col = 64 * wn + 8 * j + 2 * (lane & 3);
            *reinterpret_cast<double2*>(C + (long long)row * ldc + col) =
                make_double2(alpha * acc[i][j][0], alpha * acc[i][j][1]);
        }
    }
}

// Triangular inverse X = L^-1 (lower, row-major) by recursive doubling over 128-blocks: with X11, X22 known for the two
// halves of a pair,  X21 = -X22 (L21 X11).  One launch per product and level handles every pair of the level
// (2 ceil(log2 nb) launches, each a grid of full DMMA tiles) -- the block-column sweep of trtri() exposes at most nb-1
// CTAs per launch and took 10 of the 31 ms of a cfg1 solve (profiles/r02_cfg1_launches_v1.csv).
struct RdArgs {
    const double* L;  // Cholesky factor (lower), ld = Np
    double* X;        // inverse (lower), ld = Np; diagonal 128-blocks pre-filled
    double* S;        // scratch, ld = Np: T = L21 X11 at the coordinates of X21
    int Np, nb, hb;   // hb = blocks per half at this level
    int phase;        // 0: T = L21 X11, 1: X21 = -X22 T
};
__global__ void __launch_bounds__(NTHREADS, 1) k_trtri_rd(const __grid_constant__ RdArgs a) {
    extern __shared__ __align__(16) double sm[];
    const int per = a.hb * a.hb;
    const int p = blockIdx.x / per, r = blockIdx.x - p * per;
    const int ti = r / a.hb, tj = r - ti * a.hb;
    const int o = 2 * a.hb * p;
    const int h2 = min(a.hb, a.nb - o - a.hb);  // blocks in the second half (ragged last pair)
    if (ti >= h2) return;
    const long long Np = a.Np;
    const int row = o + a.hb + ti, col = o + tj;
    double acc[4][8][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
    if (a.phase == 0) {
        // T[row, col] = sum_{k = col .. o+hb-1} L[row, k] X[k, col]   (X11 lower triangular)
        const int k0 = col, k1 = o + a.hb;
        gemm_mainloop<true>(a.L + (long long)row * TB * Np + (long long)k0 * TB, Np,
                            a.X + (long long)k0 * TB * Np + (long long)col * TB, Np, (k1 - k0) * (TB / KC), sm, acc);
        store_tile(a.S + (long long)row * TB * Np + (long long)col * TB, Np, 1.0, acc);
    } else {
        // X[row, col] = - sum_{k = o+hb .. row} X[row, k] T[k, col]   (X22 lower triangular)
        const int k0 = o + a.hb, k1 = row + 1;
        gemm_mainloop<true>(a.X + (long long)row * TB * Np + (long long)k0 * TB, Np,
                            a.S + (long long)k0 * TB * Np + (long long)col * TB, Np, (k1 - k0) * (TB / KC), sm, acc);
        store_tile(a.X + (long long)row * TB * Np + (long long)col * TB, Np, -1.0, acc);
    }
}

// X diagonal 128-blocks <- the per-block inverses the factorisation kept (Linv, ld 128)
__global__ void __launch_bounds__(256) k_copy_diag_inv(const double* __restrict__ Linv, double* __restrict__ X, int Np) {
    const int kb = blockIdx.x;
    for (int idx = threadIdx.x; idx < TB * TB / 2; idx += 256) {
        const int r = idx >> 6, c2 = (idx & 63) * 2;
        *reinterpret_cast<double2*>(X + (long long)(kb * TB + r) * Np + kb * TB + c2) =
            *reinterpret_cast<const double2*>(Linv + (long long)kb * TB * TB + r * TB + c2);
    }
}

// C tile = A[128 x K] * B[128 x K]' (both row-major, K contiguous)
enum { NT_TRI = 1, NT_SYRK = 2 };
struct NtArgs {
    const double* A; long long lda;
    const double* B; long long ldb;
    double* C; long long ldc;
    int mt, nt, mode;
    long long K, Ksplit;
};
__global__ void __launch_bounds__(NTHREADS, 1) k_gemm_nt(const __grid_constant__ NtArgs a) {
    extern __shared__ __align__(16) double sm[];
    int I, J;
    long long Kend;
    if (a.mode == NT_TRI) {  // Q1' = L^-1 [A']: row block I of the lower-triangular L^-1 has (I+1)*128 columns; long tiles first
        const int t = blockIdx.x;
        I = a.mt - 1 - t / a.nt;
        J = t % a.nt;
        Kend = (long long)(I + 1) * TB;
    } else {  // G2 = Q1'Q1, lower tiles; the ridge block of row block J ends at column Ksplit + (J+1)*128.  Longest tiles
              // (largest J) first: block columns from the last one backwards
        int cidx, ridx;
        tile_ij(blockIdx.x, cidx, ridx);
        J = a.nt - 1 - cidx;
        I = J + ridx;
        Kend = a.Ksplit + (long long)(J + 1) * TB;
        if (Kend > a.K) Kend = a.K;
    }
    double acc[4][8][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
    gemm_mainloop<false>(a.A + (long long)I * TB * a.lda, a.lda, a.B + (long long)J * TB * a.ldb, a.ldb, (int)(Kend / KC),
                         sm, acc);
    store_tile(a.C + (long long)I * TB * a.ldc + (long long)J * TB, a.ldc, 1.0, acc);
}

// out[i] = sum_{s in [s0(i), len)} Mx[i][s] v[s], one warp per row; from_diag: s0 = first column of row i's 128-tile
__global__ void __launch_bounds__(256) k_gemv_rows(const double* __restrict__ Mx, long long ld, int nrows,
                                                   const double* __restrict__ v, long long len, int from_diag,
                                                   double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= nrows) return;
    const double* row = Mx + (long long)i * ld;
    double s0 = 0.0, s1 = 0.0;
    long long s = (from_diag ? (long long)(i & ~127) : 0) + lane;
    for (; s + 32 < len; s += 64) {
        s0 = fma(row[s], v[s], s0);
        s1 = fma(row[s + 32], v[s + 32], s1);
    }
    if (s < len) s0 = fma(row[s], v[s], s0);
    s0 += s1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s0 += __shfl_xor_sync(0xffffffffu, s0, o);
    if (lane == 0) out[i] = s0;
}

// dual (sample-space) Gram: diagonal += lam^2 on the N real samples, unit diagonal on the padding rows
__global__ void k_diag_dual(double* __restrict__ Gd, long long Nr, long long N, double lam2) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= Nr) return;
    double* g = Gd + s * Nr + s;
    *g = s < N ? *g + lam2 : 1.0;
}
// out[0] = min_i L[i][i]^2, out[1] = max_i L[i][i]^2 over the first n rows of a factor with leading dimension ld
__global__ void __launch_bounds__(256) k_pivot_range(const double* __restrict__ L, long long ld, long long n,
                                                     double* __restrict__ out) {
    __shared__ double r0[256], r1[256];
    double lo = 1.0e300, hi = 0.0;
    for (long long i = threadIdx.x; i < n; i += 256) {
        const double l = L[i * ld + i], p = l * l;
        lo = fmin(lo, p);
        hi = fmax(hi, p);
    }
    r0[threadIdx.x] = lo;
    r1[threadIdx.x] = hi;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) {
            r0[threadIdx.x] = fmin(r0[threadIdx.x], r0[threadIdx.x + s]);
            r1[threadIdx.x] = fmax(r1[threadIdx.x], r1[threadIdx.x + s]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = r0[0];
        out[1] = r1[0];
    }
}
// out[p] = sum_s Mx[s][p] v[s]  (column sums over `rows` rows; coalesced across p), grid.y splits the rows, partials summed
// in fixed order by the caller's second pass (k_colsum_finish)
__global__ void __launch_bounds__(256) k_gemv_cols(const double* __restrict__ Mx, long long ld, long long rows, int ncols,
                                                   const double* __restrict__ v, double* __restrict__ part) {
    const int p = blockIdx.x * 256 + threadIdx.x;
    const long long per = (rows + gridDim.y - 1) / gridDim.y;
    const long long s0 = blockIdx.y * per, s1 = s0 + per < rows ? s0 + per : rows;
    if (p >= ncols) return;
    double a0 = 0.0, a1 = 0.0;
    long long s = s0;
    for (; s + 1 < s1; s += 2) {
        a0 = fma(Mx[s * ld + p], v[s], a0);
        a1 = fma(Mx[(s + 1) * ld + p], v[s + 1], a1);
    }
    if (s < s1) a0 = fma(Mx[s * ld + p], v[s], a0);
    part[(long long)blockIdx.y * ncols + p] = a0 + a1;
}
__global__ void k_colsum_finish(const double* __restrict__ part, int nparts, int ncols, double* __restrict__ out) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= ncols) return;
    double t = 0.0;
    for (int q = 0; q < nparts; q++) t += part[(long long)q * ncols + p];
    out[p] = t;
}
// r <- r - lam2 * w (first n entries)
__global__ void k_axpy_neg(double* __restrict__ r, const double* __restrict__ w, double lam2, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) r[i] = fma(-lam2, w[i], r[i]);
}

// g <- A'r - lam^2 x on the real columns, 0 on the dummies
__global__ void k_csne_rhs(double* __restrict__ g, const double* __restrict__ x, double lam2, int Np, int ncc,
                           int zero_first) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= Np) return;
    g[p] = is_dummy_col(p, ncc, zero_first) ? 0.0 : g[p] - lam2 * x[p];
}

// v = -lam x on the real columns, 0 on the dummies: the ridge rows of [y; 0] - [A; lam I] x
__global__ void k_ridge_resid(double* __restrict__ v, const double* __restrict__ x, double lam, int Np, int ncc,
                              int zero_first) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= Np) return;
    v[p] = is_dummy_col(p, ncc, zero_first) ? 0.0 : -lam * x[p];
}

// x += dx; out = {|dx|^2, |x|^2}   (one CTA, fixed summation order)
__global__ void __launch_bounds__(1024) k_axpy_norms(double* __restrict__ x, const double* __restrict__ dx, int Np,
                                                     double* __restrict__ out) {
    __shared__ double r0[1024], r1[1024];
    double a = 0.0, b = 0.0;
    for (int p = threadIdx.x; p < Np; p += 1024) {
        const double d = dx[p], v = x[p] + d;
        x[p] = v;
        a = fma(d, d, a);
        b = fma(v, v, b);
    }
    r0[threadIdx.x] = a;
    r1[threadIdx.x] = b;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) {
            r0[threadIdx.x] += r0[threadIdx.x + s];
            r1[threadIdx.x] += r1[threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[0] = r0[0];
        out[1] = r1[0];
    }
}

// out[0] = min over the real columns of L[i][i]^2 (the pivots of the factorisation)
__global__ void __launch_bounds__(256) k_min_pivot(const double* __restrict__ L, int Np, int ncc, int zero_first,
                                                   double* __restrict__ out) {
    __shared__ double red[256];
    double m = 1.0e300;
    for (int i = threadIdx.x; i < Np; i += 256)
        if (!is_dummy_col(i, ncc, zero_first)) {
            const double l = L[(long long)i * Np + i];
            m = fmin(m, l * l);
        }
    red[threadIdx.x] = m;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] = fmin(red[threadIdx.x], red[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = red[0];
}

// md[1] = max(ridge, scale * md[0])
__global__ void k_set_shift(double* md, double ridge, double scale) { md[1] = fmax(ridge, scale * md[0]); }

// ---- total least squares (tls_spectral, src/lsfft.jl:87-99) ----
// out[0] = sum v[i]^2   (one CTA, fixed order)
__global__ void __launch_bounds__(1024) k_sumsq(const double* __restrict__ v, long long n, double* __restrict__ out) {
    __shared__ double red[1024];
    double a = 0.0;
    for (long long i = threadIdx.x; i < n; i += 1024) a = fma(v[i], v[i], a);
    red[threadIdx.x] = a;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = red[0];
}

// One step of inverse iteration on the bordered matrix [[M, b], [b', c]] (M = G + shift I factorised, c = y'y + shift):
// in : z = M^-1 u, g = M^-1 b, the previous iterate (u, w) and sc = {c, -, -, w}
// out: (u, w) <- normalised solution of the bordered system, sc[2] = |change|^2 (sign-aligned), sc[3] = w
__global__ void __launch_bounds__(1024) k_tls_update(const double* __restrict__ z, const double* __restrict__ g,
                                                     const double* __restrict__ b, double* __restrict__ u, int Np,
                                                     double* __restrict__ sc) {
    __shared__ double r0[1024], r1[1024];
    const int tid = threadIdx.x;
    double bz = 0.0, bg = 0.0;
    for (int i = tid; i < Np; i += 1024) {
        bz = fma(b[i], z[i], bz);
        bg = fma(b[i], g[i], bg);
    }
    r0[tid] = bz;
    r1[tid] = bg;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if (tid < s) {
            r0[tid] += r0[tid + s];
            r1[tid] += r1[tid + s];
        }
        __syncthreads();
    }
    const double schur = sc[0] - r1[0];          // c - b' M^-1 b  (> 0: the shifted bordered matrix is SPD)
    const double q = (sc[3] - r0[0]) / schur;    // last component of the solve
    __syncthreads();
    double nn = 0.0;
    for (int i = tid; i < Np; i += 1024) {
        const double p = z[i] - g[i] * q;
        nn = fma(p, p, nn);
    }
    r0[tid] = nn;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if (tid < s) r0[tid] += r0[tid + s];
        __syncthreads();
    }
    const double inv = 1.0 / sqrt(r0[0] + q * q);
    const double sgn = (q * sc[3] < 0.0) ? -1.0 : 1.0;  // keep the sign of the last component: v and -v are the same vector
    __syncthreads();
    double ch = 0.0;
    for (int i = tid; i < Np; i += 1024) {
        const double p = sgn * (z[i] - g[i] * q) * inv;
        const double d = p - u[i];
        ch = fma(d, d, ch);
        u[i] = p;
    }
    r1[tid] = ch;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if (tid < s) r1[tid] += r1[tid + s];
        __syncthreads();
    }
    if (tid == 0) {
        const double wn = sgn * q * inv, dw = wn - sc[3];
        sc[2] = r1[0] + dw * dw;
        sc[3] = wn;
    }
}

// start vector [g; -1] / |.| and c = y'y + shift
__global__ void __launch_bounds__(1024) k_tls_init(const double* __restrict__ g, double* __restrict__ u, int Np,
                                                   double* __restrict__ sc, const double* __restrict__ shift) {
    __shared__ double red[1024];
    double a = 0.0;
    for (int i = threadIdx.x; i < Np; i += 1024) a = fma(g[i], g[i], a);
    red[threadIdx.x] = a;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    const double inv = 1.0 / sqrt(red[0] + 1.0);
    for (int i = threadIdx.x; i < Np; i += 1024) u[i] = g[i] * inv;
    if (threadIdx.x == 0) {
        sc[0] += shift[0];
        sc[2] = 1.0;
        sc[3] = -inv;
    }
}

// x = -u / w on the real columns
__global__ void k_tls_finish(const double* __restrict__ u, const double* __restrict__ sc, int Np, double* __restrict__ x) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < Np) x[p] = -u[p] / sc[3];
}

int adjoint_apply(lpvs_ctx* c, const OpArgs& op, int Np, const double* d_r, double* d_out /* [2][Np] */) {
    // b = A' r through the rhs kernel of the Gram pass, split over samples so the grid fills the GPU
    const int nblk = Np / TB;
    long long want = std::max<long long>(1, (2LL * c->sms + nblk - 1) / nblk);
    long long nsplit = std::min<long long>(want, std::max<long long>(1, op.N / 256));
    long long n_split = (op.N + nsplit - 1) / nsplit;
    n_split = (n_split + KC - 1) / KC * KC;
    const int nprob = (int)((op.N + n_split - 1) / n_split);
    GramArgs g{};
    g.t = op.t;
    g.y = d_r;
    g.u = nullptr;
    g.W = nullptr;
    g.w_abs = 1;
    g.start0 = 0;
    g.hop = n_split;
    g.n = (int)n_split;
    g.s_end = op.N;
    g.ncc = op.ncc;
    g.nblk = nblk;
    g.nrhs = 1;
    g.tbl_base = 0;
    g.tbl_ns = op.tbl_ns;
    g.f = op.f;
    g.E = op.E;
    g.Kt = op.Kt;
    g.lpv_nf = op.lpv_nf;
    g.gscale = 1.0;
    g.bscale = op.mode == GRAM_DIRECT ? op.dd : 1.0;
    if (nprob == 1) {
        g.B = d_out;
        g.strideB = 0;
        c->launches += launch_gram_rhs(op.mode, g, 1, c->st);
        return LPVS_OK;
    }
    double* parts = ws<double>(c, BUF_PART, (size_t)nprob * 2 * Np);
    if (!parts) return fail(c, LPVS_E_NOMEM, "out of device memory (adjoint partials)");
    g.B = parts;
    g.strideB = 2LL * Np;
    c->launches += launch_gram_rhs(op.mode, g, nprob, c->st);
    reduce_parts(c, d_out, parts, Np, 2LL * Np, nprob, 0);
    return LPVS_OK;
}

}  // namespace

// tls_spectral (src/lsfft.jl:87-99): x = -V[1:n, n+1] / V[n+1, n+1], V the right singular vectors of [A y], i.e. the
// eigenvector of the smallest eigenvalue of [A y]'[A y] = [[G, b], [b', y'y]] -- the Gram pass already produces G and b.
// Inverse iteration with the Cholesky factor of G + shift I through the bordered (Schur complement) solve; start vector
// [x_LS; -1].  Converges at (lambda_1 + shift) / (lambda_2 + shift) per step; *iters_out = steps taken.  Like every
// Gram-based method this resolves sigma_min([A y]) down to ~1e-8 sigma_max: the well-conditioned regime of the north_star.
int tls_solve(lpvs_ctx* c, int Np, int ncc, int zero_first, const double* d_y, long long N, double* d_G, double* d_B,
              int* iters_out) {
    cudaStream_t st = c->st;
    const int nb = Np / TB;
    const long long NN = (long long)Np * Np;
    const int nreal = 2 * ncc - zero_first;
    int rc;
    double* d_md = ws<double>(c, BUF_SUMS, 8);               // [0] max diag, [1] shift, [4..7] = sc: c, -, change, w
    double* d_v = ws<double>(c, BUF_LSQ_V, (size_t)5 * Np);  // b | g = M^-1 b | u | z (2 Np: trsv layout)
    if (!d_md || !d_v) return fail(c, LPVS_E_NOMEM, "out of device memory (TLS vectors)");
    double* d_sc = d_md + 4;
    double *d_b = d_v, *d_g = d_v + Np, *d_u = d_v + 2 * Np, *d_z = d_v + 3 * Np;
    LPVS_CU(c, cudaMemcpyAsync(d_b, d_B, sizeof(double) * Np, cudaMemcpyDeviceToDevice, st));
    launch_max_diag(d_G, NN, Np, ncc, zero_first, d_md, 1, st);
    k_set_shift<<<1, 1, 0, st>>>(d_md, 0.0, (double)(nreal + 1) * EPS);
    c->launches += 2;
    int pinfo = 0;
    if ((rc = factor_solve(c, ncc, zero_first, Np, d_G, d_B, 1, 0.0, 1, &pinfo, nullptr, 0.0, d_md + 1))) return rc;
    LPVS_CU(c, cudaMemcpyAsync(d_g, d_B, sizeof(double) * Np, cudaMemcpyDeviceToDevice, st));
    k_sumsq<<<1, 1024, 0, st>>>(d_y, N, d_sc);
    k_tls_init<<<1, 1024, 0, st>>>(d_g, d_u, Np, d_sc, d_md + 1);
    c->launches += 2;
    LPVS_CU(c, cudaStreamSynchronize(st));
    if (pinfo) return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown at internal pivot %d (TLS)", pinfo);
    CholArgs ca{};
    ca.G = d_G;
    ca.strideG = NN;
    ca.Linv = ws<double>(c, BUF_LINV, (size_t)nb * TB * TB);
    ca.strideLinv = (long long)nb * TB * TB;
    ca.info = ws<int>(c, BUF_INFO, 1);
    ca.Np = Np;
    ca.nb = nb;
    int it = 0;
    for (it = 1; it <= 300; it++) {
        LPVS_CU(c, cudaMemcpyAsync(d_z, d_u, sizeof(double) * Np, cudaMemcpyDeviceToDevice, st));
        launch_trsv(ca, d_z, 2LL * Np, 1, 1, st, false, trsv_flags(c, nb));
        k_tls_update<<<1, 1024, 0, st>>>(d_z, d_g, d_b, d_u, Np, d_sc);
        c->launches += 2;
        double ch = 0.0;
        LPVS_CU(c, cudaMemcpyAsync(&ch, d_sc + 2, sizeof(double), cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaStreamSynchronize(st));
        if (!isfinite(ch) || ch <= 1e-28) break;  // |v_k - v_(k-1)| <= 1e-14 (unit vectors)
    }
    if (iters_out) *iters_out = it;
    k_tls_finish<<<(Np + 255) / 256, 256, 0, st>>>(d_u, d_sc, Np, d_B);
    c->launches++;
    return LPVS_OK;
}

namespace {
// Underdetermined problems (Nreg >= N): x = A'(A A' + lam^2 I)^-1 y -- the same ridge solution through the N x N Gram
// matrix of the ROWS.  With more functions than samples the row space is the well-conditioned side (the reference's KAT,
// 1000 x 1001, has cond(A A') = 2 against a singular A'A); the sample-space Gram matrix is one NT DMMA pass over the
// materialised regressor, and iterative refinement on the operator brings the answer to cond(A) eps.  Returns 1 when the
// factorisation is too ill-conditioned to trust (the caller falls back to the column-space path), 0 on success.
int ls_solve_dual(lpvs_ctx* c, const OpArgs& op, int Np, const double* d_y, double lam, double* d_x, int* rc_out) {
    cudaStream_t st = c->st;
    const long long N = op.N, Nr = (N + TB - 1) / TB * TB;
    const int nbd = (int)(Nr / TB), nb = Np / TB;
    const double lam2 = lam * lam;
    *rc_out = LPVS_OK;
    double* d_A = ws<double>(c, BUF_LSQ_A, (size_t)Nr * Np);
    double* d_Gd = ws<double>(c, BUF_LSQ_G2, (size_t)std::max<long long>(Nr * Nr, (long long)Np * Np));
    double* d_w = ws<double>(c, BUF_LSQ_R, (size_t)std::max<long long>(6 * Nr, Nr + Np));  // w | r (2 Nr: trsv layout) | spare
    double* d_md = ws<double>(c, BUF_SUMS, 8);
    const int nsplit = 32;
    double* d_part = ws<double>(c, BUF_PART, (size_t)nsplit * Np);
    if (!d_A || !d_Gd || !d_w || !d_md || !d_part) {
        *rc_out = fail(c, LPVS_E_NOMEM, "out of device memory (sample-space solve of a %lld x %d problem)", N, Np);
        return 0;
    }
    static bool attr_done[64] = {};
    const size_t smem = (size_t)NT_STAGES * 2 * TILE_D * sizeof(double);
    if (!attr_done[c->device & 63]) {
        cudaFuncSetAttribute(k_gemm_nt, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_trtri_rd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_done[c->device & 63] = true;
    }
    dim3 gm((unsigned)((Nr + 3) / 4), nb);
    k_materialize<<<gm, 256, 0, st>>>(op, d_A, Np, Nr);
    NtArgs t{};
    t.A = d_A; t.lda = Np;
    t.B = d_A; t.ldb = Np;
    t.C = d_Gd; t.ldc = Nr;
    t.mt = nbd; t.nt = nbd; t.mode = NT_SYRK;
    t.K = Np; t.Ksplit = Np;
    k_gemm_nt<<<nbd * (nbd + 1) / 2, NTHREADS, smem, st>>>(t);
    k_diag_dual<<<(unsigned)((Nr + 255) / 256), 256, 0, st>>>(d_Gd, Nr, N, lam2);
    c->launches += 3;
    CholArgs ca{};
    ca.G = d_Gd;
    ca.strideG = Nr * Nr;
    ca.Linv = ws<double>(c, BUF_LINV, (size_t)std::max(nbd, nb) * TB * TB);
    ca.strideLinv = (long long)nbd * TB * TB;
    ca.info = ws<int>(c, BUF_INFO, 1);
    ca.Np = (int)Nr;
    ca.nb = nbd;
    if (!ca.Linv || !ca.info) {
        *rc_out = fail(c, LPVS_E_NOMEM, "out of device memory (factor workspace)");
        return 0;
    }
    cudaMemsetAsync(ca.info, 0, sizeof(int), st);
    c->launches += potrf(ca, 1, c->sms, st, &c->la);
    k_pivot_range<<<1, 256, 0, st>>>(d_Gd, Nr, N, d_md + 4);
    c->launches++;
    int pinfo = 0;
    double pr[2] = {0.0, 0.0};
    cudaMemcpyAsync(&pinfo, ca.info, sizeof(int), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(pr, d_md + 4, sizeof pr, cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) {
        *rc_out = fail(c, LPVS_E_CUDA, "sample-space factorisation failed");
        return 0;
    }
    // iterative refinement converges while cond(A A' + lam^2 I) eps << 1; the pivot ratio is a (lower) estimate of that cond
    if (pinfo != 0 || !(pr[0] > 1e-10 * pr[1])) return 1;
    double* d_r = d_w + Nr;  // [2][Nr] right-hand side / solution of the triangular solves
    cudaMemsetAsync(d_w, 0, sizeof(double) * 3 * Nr, st);
    cudaMemsetAsync(d_x, 0, sizeof(double) * Np, st);
    double prev = 0.0;
    bool ok = false;
    for (int step = 0; step < 6; step++) {
        // r = y - A x - lam^2 w  (first step: x = w = 0 -> r = y)
        k_op_apply<<<(unsigned)((N + 31) / 32), 256, 0, st>>>(op, d_x, d_y, d_r);
        k_axpy_neg<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(d_r, d_w, lam2, N);
        if (Nr > N) cudaMemsetAsync(d_r + N, 0, sizeof(double) * (Nr - N), st);
        launch_trsv(ca, d_r, 2 * Nr, 1, 1, st, false, trsv_flags(c, nbd));
        k_axpy_norms<<<1, 1024, 0, st>>>(d_w, d_r, (int)Nr, d_md + 2);  // w += dw
        dim3 gc((Np + 255) / 256, nsplit);
        k_gemv_cols<<<gc, 256, 0, st>>>(d_A, Np, N, Np, d_w, d_part);
        k_colsum_finish<<<(Np + 255) / 256, 256, 0, st>>>(d_part, nsplit, Np, d_x);  // x = A' w
        c->launches += 6;
        double h[2] = {0.0, 0.0};
        cudaMemcpyAsync(h, d_md + 2, sizeof h, cudaMemcpyDeviceToHost, st);
        if (cudaStreamSynchronize(st) != cudaSuccess) {
            *rc_out = fail(c, LPVS_E_CUDA, "sample-space refinement failed");
            return 0;
        }
        if (!(isfinite(h[0]) && isfinite(h[1]))) return 0;  // NaN inputs: the caller's finite check reports the cause
        const double rel = h[1] > 0.0 ? sqrt(h[0] / h[1]) : 0.0;
        if (step > 0 && rel <= 1e-12) {
            ok = true;
            break;
        }
        if (step > 1 && rel > 0.25 * prev) break;  // not contracting: too ill-conditioned for this side
        prev = rel;
    }
    return ok ? 0 : 1;
}
}  // namespace

int ls_solve_accurate(lpvs_ctx* c, const OpArgs& op, int Np, int zero_first, const double* d_y, double* d_G, double* d_B,
                      double lam, const std::function<int()>& regram, int* info) {
    cudaStream_t st = c->st;
    const int nb = Np / TB, ncc = op.ncc;
    const long long NN = (long long)Np * Np, N = op.N;
    const int nreal = 2 * ncc - zero_first;
    const double lam2 = lam * lam;
    int rc;
    if (info) *info = 0;
    double* d_md = ws<double>(c, BUF_SUMS, 8);  // [0] max diag, [1] shift, [2..3] norms
    double* d_r = ws<double>(c, BUF_LSQ_R, (size_t)std::max<long long>(N, Np));
    double* d_g = ws<double>(c, BUF_LSQ_V, (size_t)4 * Np);
    if (!d_md || !d_r || !d_g) return fail(c, LPVS_E_NOMEM, "out of device memory (LS refinement vectors)");

    // ---- 0. more functions than samples: the sample-space (dual) solve; falls through when that side is ill-conditioned ----
    if (nreal >= N && lam > 0.0) {
        int rcd = LPVS_OK;
        const int fallback = ls_solve_dual(c, op, Np, d_y, lam, d_g, &rcd);  // x into scratch: d_B (A'y) survives a fallback
        if (rcd) return rcd;
        if (!fallback) {
            LPVS_CU(c, cudaMemcpyAsync(d_B, d_g, sizeof(double) * Np, cudaMemcpyDeviceToDevice, st));
            LPVS_CU(c, cudaStreamSynchronize(st));
            if (info) *info = LPVS_INFO_DUAL;
            return LPVS_OK;
        }
    }
    // ---- 1. one factorisation: L L' = G~ + max(lam^2, n eps max diag) I ----
    int pinfo = 0;
    double mult = 1.0;
    double hmin[2] = {0.0, 0.0};  // smallest squared pivot of the factor, the shift
    for (int attempt = 0;; attempt++) {
        launch_max_diag(d_G, NN, Np, ncc, zero_first, d_md, 1, st);
        k_set_shift<<<1, 1, 0, st>>>(d_md, lam2, mult * (double)nreal * EPS);
        c->launches += 2;
        // attempt 0: plain; a breakdown is first answered with the SAME shift and refined TRSM tiles (attempt 1), and only then
        // with larger shifts -- the shift bounds lam^2 / shift, the smallest eigenvalue the QR path's G2 has to resolve
        if ((rc = factor_solve(c, ncc, zero_first, Np, d_G, d_B, 1, 0.0, 1, &pinfo, nullptr, 0.0, d_md + 1, attempt > 0)))
            return rc;
        k_min_pivot<<<1, 256, 0, st>>>(d_G, Np, ncc, zero_first, d_md + 4);
        c->launches++;
        LPVS_CU(c, cudaMemcpyAsync(&hmin[0], d_md + 4, sizeof(double), cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaMemcpyAsync(&hmin[1], d_md + 1, sizeof(double), cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaStreamSynchronize(st));
        if (pinfo == 0) break;
        if (attempt == 4 || !isfinite(mult)) {
            if (info) *info = pinfo;
            return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown at internal pivot %d even with a %g n eps shift", pinfo, mult);
        }
        if (attempt > 0) mult *= 32.0;  // the shift only conditions the preconditioner, not the solution
        if ((rc = regram())) return rc;
    }
    double* d_x = d_B;  // x0 = (G~ + shift)^-1 A'y
    // Pivots at the level of the shift mean directions with sigma^2 <~ shift, where the refinement contracts by shift / (sigma^2
    // + shift) ~ 1 per step: go straight to the QR path (which is also exact where the refinement would have converged).
    const bool hopeless = hmin[0] < 8.0 * hmin[1];

    CholArgs ca{};
    ca.G = d_G;
    ca.strideG = NN;
    ca.Linv = ws<double>(c, BUF_LINV, (size_t)nb * TB * TB);
    ca.strideLinv = (long long)nb * TB * TB;
    ca.info = ws<int>(c, BUF_INFO, 1);
    ca.Np = Np;
    ca.nb = nb;

    // ---- 2. corrected semi-normal equations on the reference-rounded operator ----
    double prev = 0.0;
    bool converged = false;
    for (int step = 1; step <= 8 && !hopeless; step++) {
        k_op_apply<<<(unsigned)((N + 31) / 32), 256, 0, st>>>(op, d_x, d_y, d_r);
        c->launches++;
        if ((rc = adjoint_apply(c, op, Np, d_r, d_g))) return rc;
        k_csne_rhs<<<(Np + 255) / 256, 256, 0, st>>>(d_g, d_x, lam2, Np, ncc, zero_first);
        launch_trsv(ca, d_g, 2LL * Np, 1, 1, st, false, trsv_flags(c, nb));
        k_axpy_norms<<<1, 1024, 0, st>>>(d_x, d_g, Np, d_md + 2);
        c->launches += 3;
        double h[2] = {0.0, 0.0};
        LPVS_CU(c, cudaMemcpyAsync(h, d_md + 2, sizeof h, cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaStreamSynchronize(st));
        if (!(isfinite(h[0]) && isfinite(h[1]))) break;  // NaN inputs: the caller's finite check reports the cause
        const double rel = h[1] > 0.0 ? sqrt(h[0] / h[1]) : 0.0;
#ifdef LPVS_DEBUG_LSQ
        fprintf(stderr, "[lsq] refinement step %d: |dx|/|x| = %.3e (min pivot^2 %.3e, shift %.3e)\n", step, rel, hmin[0], hmin[1]);
#endif
        // A step that moved x by <= 1e-11 with a contraction <= 0.05 per step leaves an error below 1e-12: well inside the
        // 1e-9 parity bar, and above the 1e-13 level at which the steps only reshuffle rounding noise.
        if (rel <= 1e-11) {
            converged = true;
            break;
        }
        // contraction too slow -- cond(A)^2 eps is not small against the shift (the first step's size is about the
        // contraction factor itself): the QR path takes over
        if (rel > 0.05 * (step == 1 ? 1.0 : prev)) break;
        prev = rel;
    }
    if (converged) return LPVS_OK;

    // ---- 3. shifted CholeskyQR on the materialised regressor ----
    if (info) *info = LPVS_INFO_QR;
    const long long Nr = (N + TB - 1) / TB * TB, Mrows = Nr + Np;
    double* d_Y = ws<double>(c, BUF_LSQ_Y, (size_t)NN);
    double* d_Li = ws<double>(c, BUF_LSQ_LI, (size_t)NN);
    double* d_A = ws<double>(c, BUF_LSQ_A, (size_t)Nr * Np);
    double* d_Bt = ws<double>(c, BUF_LSQ_BT, (size_t)Np * Mrows);
    double* d_G2 = ws<double>(c, BUF_LSQ_G2, (size_t)NN);
    if (!d_Y || !d_Li || !d_A || !d_Bt || !d_G2)
        return fail(c, LPVS_E_NOMEM, "out of device memory (QR path of a rank-deficient %d x %d problem)", (int)N, nreal);
    static bool attr_done[64] = {};
    const size_t smem = (size_t)NT_STAGES * 2 * TILE_D * sizeof(double);
    if (!attr_done[c->device & 63]) {
        cudaFuncSetAttribute(k_gemm_nt, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_trtri_rd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_done[c->device & 63] = true;
    }
    {
        // X = L^-1 into d_Li by recursive doubling (d_G2 is free until the SYRK below: scratch for T)
        LPVS_CU(c, cudaMemsetAsync(d_Li, 0, sizeof(double) * NN, st));
        k_copy_diag_inv<<<nb, 256, 0, st>>>(ca.Linv, d_Li, Np);
        c->launches++;
        RdArgs rd{};
        rd.L = d_G;
        rd.X = d_Li;
        rd.S = d_G2;
        rd.Np = Np;
        rd.nb = nb;
        for (int hb = 1; hb < nb; hb <<= 1) {
            const int npairs = (nb + 2 * hb - 1) / (2 * hb);
            rd.hb = hb;
            for (rd.phase = 0; rd.phase < 2; rd.phase++) {
                k_trtri_rd<<<npairs * hb * hb, NTHREADS, smem, st>>>(rd);
                c->launches++;
            }
        }
        dim3 grid(Np / 32, Np / 32);
        k_transpose_linv<<<grid, 256, 0, st>>>(d_Li, Np, ncc, zero_first, lam, d_Y, d_Bt, Mrows, Nr);
        dim3 gm((unsigned)((Nr + 3) / 4), nb);
        k_materialize<<<gm, 256, 0, st>>>(op, d_A, Np, Nr);
        c->launches += 2;
    }
    NtArgs t1{};
    t1.A = d_Li; t1.lda = Np;
    t1.B = d_A; t1.ldb = Np;
    t1.C = d_Bt; t1.ldc = Mrows;
    t1.mt = nb; t1.nt = (int)(Nr / TB); t1.mode = NT_TRI;
    t1.K = Np; t1.Ksplit = 0;
    k_gemm_nt<<<t1.mt * t1.nt, NTHREADS, smem, st>>>(t1);
    NtArgs t2{};
    t2.A = d_Bt; t2.lda = Mrows;
    t2.B = d_Bt; t2.ldb = Mrows;
    t2.C = d_G2; t2.ldc = Np;
    t2.mt = nb; t2.nt = nb; t2.mode = NT_SYRK;
    t2.K = Mrows; t2.Ksplit = Nr;
    k_gemm_nt<<<nb * (nb + 1) / 2, NTHREADS, smem, st>>>(t2);
#ifdef LPVS_DEBUG_LSQ
    if (const char* dump = getenv("LPVS_DEBUG_DUMP")) {  // developer build only: the QR path's matrices for offline comparison
        cudaStreamSynchronize(st);
        std::vector<double> hb((size_t)std::max<long long>(NN, (long long)Np * Mrows));
        if (FILE* fp = fopen(dump, "wb")) {
            long long hdr[4] = {Np, Mrows, Nr, N};
            fwrite(hdr, sizeof(long long), 4, fp);
            for (const double* src : {(const double*)d_G, (const double*)d_Li, (const double*)d_G2}) {
                cudaMemcpy(hb.data(), src, sizeof(double) * NN, cudaMemcpyDeviceToHost);
                fwrite(hb.data(), sizeof(double), (size_t)NN, fp);
            }
            cudaMemcpy(hb.data(), d_Bt, sizeof(double) * Np * Mrows, cudaMemcpyDeviceToHost);
            fwrite(hb.data(), sizeof(double), (size_t)Np * Mrows, fp);
            fclose(fp);
        }
    }
#endif
    // c = Q1' [y; 0]
    LPVS_CU(c, cudaMemsetAsync(d_g, 0, sizeof(double) * 4 * Np, st));
    k_gemv_rows<<<(Np + 7) / 8, 256, 0, st>>>(d_Bt, Mrows, Np, d_y, N, 0, d_g);
    c->launches += 3;
    if ((rc = factor_solve(c, ncc, zero_first, Np, d_G2, d_g, 1, 0.0, 1, &pinfo))) return rc;
    LPVS_CU(c, cudaStreamSynchronize(st));
    if (pinfo) {  // once more with refined TRSM tiles (G2 has eigenvalues down to lam^2 / shift)
        k_gemm_nt<<<nb * (nb + 1) / 2, NTHREADS, smem, st>>>(t2);
        LPVS_CU(c, cudaMemsetAsync(d_g, 0, sizeof(double) * 4 * Np, st));
        k_gemv_rows<<<(Np + 7) / 8, 256, 0, st>>>(d_Bt, Mrows, Np, d_y, N, 0, d_g);
        c->launches += 2;
        if ((rc = factor_solve(c, ncc, zero_first, Np, d_G2, d_g, 1, 0.0, 1, &pinfo, nullptr, 0.0, nullptr, true))) return rc;
    }
    // x = L^-T z = Y z
    k_gemv_rows<<<(Np + 7) / 8, 256, 0, st>>>(d_Y, Np, Np, d_g, Np, 1, d_x);
    c->launches++;
    LPVS_CU(c, cudaStreamSynchronize(st));
    if (pinfo) {
        // Last resort.  The blocked factorisation applies its diagonal blocks through explicit inverses, so a matrix with MANY
        // null directions (Nreg well above N, with near-coincident sample times making the row space ill-conditioned too) needs
        // a shift ~1e-9 max diag to factorise, and lam^2 / shift then falls below what G2 can resolve.  The reference's SVD
        // still returns a (noise-dominated, |x| ~ |y| / lam) vector there; this library returns the shift-regularised solution
        // (G~ + shift I)^-1 A'y and says so: *info = LPVS_INFO_JITTER.
        if ((rc = regram())) return rc;
        launch_max_diag(d_G, NN, Np, ncc, zero_first, d_md, 1, st);
        k_set_shift<<<1, 1, 0, st>>>(d_md, lam2, mult * (double)nreal * EPS);
        c->launches += 2;
        if ((rc = factor_solve(c, ncc, zero_first, Np, d_G, d_B, 1, 0.0, 1, &pinfo, nullptr, 0.0, d_md + 1))) return rc;
        LPVS_CU(c, cudaStreamSynchronize(st));
        if (pinfo) {
            if (info) *info = pinfo;
            return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown at internal pivot %d (rank-deficient problem, last resort)", pinfo);
        }
        if (info) *info = LPVS_INFO_JITTER;
        return LPVS_OK;
    }
    // Refinement in the Q1 coordinates: dz = G2^-1 Q1'([y; 0] - [A; lam I] x), x += Y dz.  G2 is well conditioned, so this is
    // an (almost) exact Newton step in EVERY direction -- including the ones A cannot see, where the Cholesky solve of G2
    // leaves noise of eps |y| sqrt(shift) / lam^2 (a QR would leave eps |y| / lam).
    double* d_v = ws<double>(c, BUF_LSQ_R, (size_t)Mrows);
    if (!d_v) return fail(c, LPVS_E_NOMEM, "out of device memory (QR refinement)");
    CholArgs c2 = ca;
    c2.G = d_G2;
    c2.Y = nullptr;
    double* d_dx = d_g + 2 * Np;
    for (int step = 0; step < 2; step++) {
        k_op_apply<<<(unsigned)((N + 31) / 32), 256, 0, st>>>(op, d_x, d_y, d_v);
        if (Nr > N) LPVS_CU(c, cudaMemsetAsync(d_v + N, 0, sizeof(double) * (Nr - N), st));
        k_ridge_resid<<<(Np + 255) / 256, 256, 0, st>>>(d_v + Nr, d_x, lam, Np, ncc, zero_first);
        k_gemv_rows<<<(Np + 7) / 8, 256, 0, st>>>(d_Bt, Mrows, Np, d_v, Mrows, 0, d_g);
        launch_trsv(c2, d_g, 2LL * Np, 1, 1, st, false, trsv_flags(c, nb));
        k_gemv_rows<<<(Np + 7) / 8, 256, 0, st>>>(d_Y, Np, Np, d_g, Np, 1, d_dx);
        k_axpy_norms<<<1, 1024, 0, st>>>(d_x, d_dx, Np, d_md + 2);
        c->launches += 6;
        double h[2] = {0.0, 0.0};
        LPVS_CU(c, cudaMemcpyAsync(h, d_md + 2, sizeof h, cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaStreamSynchronize(st));
        // a second step only when the first one moved x by more than cond(G2)*eps can explain
        if (!(isfinite(h[0]) && isfinite(h[1])) || h[0] <= 1e-16 * h[1]) break;
    }
    return LPVS_OK;
}


// ======================================================================================================================
// ls_spectral of C channels sampled at the same times (lpvs_ls_spectral_multi).  Everything that depends only on t, W and
// f -- Gram matrix, factors, L^-1, the QR objects -- is built once; the y-dependent refinement runs C-wide.  Every kernel
// below gives each channel the same arithmetic whatever the number of channels, their order or the chunk a channel lands
// in, so a channel's bits do not depend on the other channels of the call.
namespace {

constexpr int OPM_CW = 16;  // channels per CTA of k_op_apply_multi

// R[c][s] = (Y ? Y[c][s] : 0) - sum_cc A[s,cc] X[c][p(cc)]: k_op_apply for a chunk of OPM_CW channels; each element is
// synthesised once for the chunk, each channel accumulates in k_op_apply's order (column slice per warp, then 8 partials)
__global__ void __launch_bounds__(256) k_op_apply_multi(const __grid_constant__ OpArgs a, const double* __restrict__ X,
                                                        long long ldx, const double* __restrict__ Y, long long ldy,
                                                        double* __restrict__ R, long long ldr, int C) {
    __shared__ double part[8][OPM_CW][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int c0 = blockIdx.y * OPM_CW, nc = min(OPM_CW, C - c0);
    const long long s = (long long)blockIdx.x * 32 + lane;
    const bool valid = s < a.N;
    const long long sc = valid ? s : a.N - 1;
    const double ts = a.mode == GRAM_DIRECT ? a.t[sc] : 0.0;
    double acc[OPM_CW];
#pragma unroll
    for (int j = 0; j < OPM_CW; j++) acc[j] = 0.0;
    for (int cc = w; cc < a.ncc; cc += 8) {
        const double2 v = op_elem(a, cc, sc, ts);
        const int p = (cc >> 6) * 128 + (cc & 63);
#pragma unroll
        for (int j = 0; j < OPM_CW; j++) {
            const double* x = X + (long long)(c0 + (j < nc ? j : 0)) * ldx;  // absent channels: computed, never stored
            acc[j] = fma(v.x, x[p], acc[j]);
            acc[j] = fma(v.y, x[p + 64], acc[j]);
        }
    }
#pragma unroll
    for (int j = 0; j < OPM_CW; j++) part[w][j][lane] = acc[j];
    __syncthreads();
    if (!valid) return;
    for (int j = w; j < nc; j += 8) {
        double t = 0.0;
#pragma unroll
        for (int q = 0; q < 8; q++) t += part[q][j][lane];
        R[(long long)(c0 + j) * ldr + s] = (Y ? Y[(long long)(c0 + j) * ldy + s] : 0.0) - t;
    }
}

// Skinny product out[c][i] = sum_k op(M)[i][k] V[c][k] for up to SK_CW channels per CTA, op(M)[i][k] = TRANS ? M[k][i] :
// M[i][k] (row-major, ld).  grid = (rows / 32, k splits, channel chunks): a CTA streams one 32-row x k-split slab of M once
// for all channels of its chunk through shared memory; each output is one FP64 FMA chain over its split in k order, the
// splits are summed in split order by k_skinny_reduce.  The split boundaries depend only on (rows, K), so every channel gets
// the same arithmetic whatever C.  tri = SK_LOWER / SK_UPPER skips the 32-tiles of op(M) that lie wholly outside its lower /
// upper triangle (they must hold zeros).
constexpr int SK_CW = 32, SK_FULL = 0, SK_LOWER = 1, SK_UPPER = 2;
template <bool TRANS>
__global__ void __launch_bounds__(256) k_skinny(const double* __restrict__ M, long long ld, int rows, long long K, int tri,
                                                const double* __restrict__ V, long long ldv, int C, long long kchunk,
                                                double* __restrict__ part) {
    __shared__ double Ms[32][33], Vs[SK_CW][33];
    const int tid = threadIdx.x, lx = tid & 31, ly = tid >> 5;
    const int r0 = blockIdx.x * 32, c0 = blockIdx.z * SK_CW, nc = min(SK_CW, C - c0);
    long long kb = (long long)blockIdx.y * kchunk, ke = min(K, kb + kchunk);
    if (tri == SK_LOWER) ke = min(ke, (long long)r0 + 32);
    if (tri == SK_UPPER) kb = max(kb, (long long)r0);
    double acc[SK_CW / 8];
#pragma unroll
    for (int j = 0; j < SK_CW / 8; j++) acc[j] = 0.0;
    for (long long k0 = kb; k0 < ke; k0 += 32) {
        for (int q = ly; q < 32; q += 8) {
            if (TRANS) {  // Ms[i][kk] = M[k0 + kk][r0 + i]: coalesced along i
                const long long k = k0 + q;
                Ms[lx][q] = (k < ke && r0 + lx < rows) ? M[k * ld + r0 + lx] : 0.0;
            } else {
                const long long k = k0 + lx;
                Ms[q][lx] = (k < ke && r0 + q < rows) ? M[(long long)(r0 + q) * ld + k] : 0.0;
            }
        }
        for (int q = ly; q < SK_CW; q += 8) {
            const long long k = k0 + lx;
            Vs[q][lx] = (k < ke && q < nc) ? V[(long long)(c0 + q) * ldv + k] : 0.0;
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < 32; kk++) {
            const double m = Ms[lx][kk];
#pragma unroll
            for (int j = 0; j < SK_CW / 8; j++) acc[j] = fma(m, Vs[ly + 8 * j][kk], acc[j]);
        }
        __syncthreads();
    }
    if (r0 + lx >= rows) return;
#pragma unroll
    for (int j = 0; j < SK_CW / 8; j++) {
        const int ch = ly + 8 * j;
        if (ch < nc) part[((long long)blockIdx.y * C + c0 + ch) * rows + r0 + lx] = acc[j];
    }
}
// out[c][i] = sum over splits in order; channels with active[c] == 0 are not written (active nullable = all)
__global__ void k_skinny_reduce(const double* __restrict__ part, int nsplit, int rows, int C, const int* __restrict__ active,
                                double* __restrict__ out, long long ldo) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x, ch = blockIdx.y;
    if (i >= rows || (active && !active[ch])) return;
    double t = part[(long long)ch * rows + i];
    for (int q = 1; q < nsplit; q++) t += part[((long long)q * C + ch) * rows + i];
    out[(long long)ch * ldo + i] = t;
}

// g[c] <- A'r - lam^2 x on the real columns, 0 on the dummies (k_csne_rhs per channel)
__global__ void k_csne_rhs_multi(double* __restrict__ g, const double* __restrict__ x, double lam2, int Np, int ncc,
                                 int zero_first) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= Np) return;
    const long long o = (long long)blockIdx.y * Np + p;
    g[o] = is_dummy_col(p, ncc, zero_first) ? 0.0 : g[o] - lam2 * x[o];
}
// v[c][off + p] = -lam x[c][p] on the real columns, 0 on the dummies (k_ridge_resid per channel)
__global__ void k_ridge_resid_multi(double* __restrict__ v, long long ldv, long long off, const double* __restrict__ x,
                                    double lam, int Np, int ncc, int zero_first) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= Np) return;
    const int ch = blockIdx.y;
    v[ch * ldv + off + p] = is_dummy_col(p, ncc, zero_first) ? 0.0 : -lam * x[(long long)ch * Np + p];
}
// r[c][i] <- r[c][i] - lam2 w[c][i] (first n entries)
__global__ void k_axpy_neg_multi(double* __restrict__ r, long long ldr, const double* __restrict__ w, long long ldw,
                                 double lam2, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long ch = blockIdx.y;
    r[ch * ldr + i] = fma(-lam2, w[ch * ldw + i], r[ch * ldr + i]);
}
// one CTA per channel, k_axpy_norms' order: x[c] += dx[c]; out[c] = {|dx|^2, |x|^2}.  Inactive channels are left alone.
__global__ void __launch_bounds__(1024) k_axpy_norms_multi(double* __restrict__ x, long long ldx,
                                                           const double* __restrict__ dx, long long lddx, int n,
                                                           const int* __restrict__ active, double* __restrict__ out) {
    __shared__ double r0[1024], r1[1024];
    const int ch = blockIdx.x;
    if (!active[ch]) return;
    double* xc = x + (long long)ch * ldx;
    const double* dc = dx + (long long)ch * lddx;
    double a = 0.0, b = 0.0;
    for (int p = threadIdx.x; p < n; p += 1024) {
        const double d = dc[p], v = xc[p] + d;
        xc[p] = v;
        a = fma(d, d, a);
        b = fma(v, v, b);
    }
    r0[threadIdx.x] = a;
    r1[threadIdx.x] = b;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) {
            r0[threadIdx.x] += r0[threadIdx.x + s];
            r1[threadIdx.x] += r1[threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[2 * ch] = r0[0];
        out[2 * ch + 1] = r1[0];
    }
}
}  // namespace

int skinny_apply(lpvs_ctx* c, const double* M, long long ld, bool trans, int tri, int rows, long long K, const double* V,
                 long long ldv, int C, const int* d_active, double* out, long long ldo) {
    const int rt = (rows + 31) / 32;
    // k splits: enough CTAs for two waves, each split >= 256 of k; a function of (rows, K) only
    long long nsplit = std::max<long long>(1, std::min<long long>(K / 256, (2LL * c->sms + rt - 1) / rt));
    long long kchunk = (K + nsplit - 1) / nsplit;
    kchunk = (kchunk + 31) / 32 * 32;
    nsplit = (K + kchunk - 1) / kchunk;
    if (nsplit < 1) nsplit = 1;
    double* part = ws<double>(c, BUF_MC_PART, (size_t)nsplit * C * rows);
    if (!part) return fail(c, LPVS_E_NOMEM, "out of device memory (skinny product partials)");
    dim3 grid(rt, (unsigned)nsplit, (C + SK_CW - 1) / SK_CW);
    if (trans)
        k_skinny<true><<<grid, 256, 0, c->st>>>(M, ld, rows, K, tri, V, ldv, C, kchunk, part);
    else
        k_skinny<false><<<grid, 256, 0, c->st>>>(M, ld, rows, K, tri, V, ldv, C, kchunk, part);
    k_skinny_reduce<<<dim3((rows + 255) / 256, C), 256, 0, c->st>>>(part, (int)nsplit, rows, C, d_active, out, ldo);
    c->launches += 2;
    LPVS_CU(c, cudaGetLastError());
    return LPVS_OK;
}

namespace {
void set_nt_smem(lpvs_ctx* c) {
    static bool attr_done[64] = {};
    const size_t smem = (size_t)NT_STAGES * 2 * TILE_D * sizeof(double);
    if (!attr_done[c->device & 63]) {
        cudaFuncSetAttribute(k_gemm_nt, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_trtri_rd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_done[c->device & 63] = true;
    }
}
}  // namespace

int factor_inverse(lpvs_ctx* c, const double* d_L, const double* d_diag_inv, int Np, double* d_X, double* d_S) {
    const int nb = Np / TB;
    const long long NN = (long long)Np * Np;
    set_nt_smem(c);
    const size_t smem = (size_t)NT_STAGES * 2 * TILE_D * sizeof(double);
    LPVS_CU(c, cudaMemsetAsync(d_X, 0, sizeof(double) * NN, c->st));
    k_copy_diag_inv<<<nb, 256, 0, c->st>>>(d_diag_inv, d_X, Np);
    c->launches++;
    RdArgs rd{};
    rd.L = d_L;
    rd.X = d_X;
    rd.S = d_S;
    rd.Np = Np;
    rd.nb = nb;
    for (int hb = 1; hb < nb; hb <<= 1) {
        const int npairs = (nb + 2 * hb - 1) / (2 * hb);
        rd.hb = hb;
        for (rd.phase = 0; rd.phase < 2; rd.phase++) {
            k_trtri_rd<<<npairs * hb * hb, NTHREADS, smem, c->st>>>(rd);
            c->launches++;
        }
    }
    LPVS_CU(c, cudaGetLastError());
    return LPVS_OK;
}

int llt_solve_multi(lpvs_ctx* c, const double* d_X, int n, const double* d_B, int C, const int* d_active, double* d_out,
                    double* d_tmp) {
    int rc;
    if ((rc = skinny_apply(c, d_X, n, false, SK_LOWER, n, n, d_B, n, C, nullptr, d_tmp, n))) return rc;
    return skinny_apply(c, d_X, n, true, SK_UPPER, n, n, d_tmp, n, C, d_active, d_out, n);
}

int adjoint_apply_multi(lpvs_ctx* c, const GramArgs& base, int mode, int Np, const double* d_R, long long ldr, int C,
                        double* d_out) {
    // B = A' diag(W) R for C channels, split over samples as adjoint_apply (the split depends on N and Np only)
    const int nblk = Np / TB;
    const long long N = base.s_end - base.start0;
    long long want = std::max<long long>(1, (2LL * c->sms + nblk - 1) / nblk);
    long long nsplit = std::min<long long>(want, std::max<long long>(1, N / 256));
    long long n_split = (N + nsplit - 1) / nsplit;
    n_split = (n_split + KC - 1) / KC * KC;
    const int nprob = (int)((N + n_split - 1) / n_split);
    GramArgs g = base;
    g.hop = n_split;
    g.n = (int)n_split;
    if (nprob == 1) {
        g.B = d_out;
        g.strideB = 0;
        c->launches += launch_gram_rhs_multi(mode, g, d_R, ldr, C, 1, c->st);
        return LPVS_OK;
    }
    double* parts = ws<double>(c, BUF_PART, (size_t)nprob * C * Np);
    if (!parts) return fail(c, LPVS_E_NOMEM, "out of device memory (adjoint partials of %d channels)", C);
    g.B = parts;
    g.strideB = (long long)C * Np;
    c->launches += launch_gram_rhs_multi(mode, g, d_R, ldr, C, nprob, c->st);
    reduce_parts(c, d_out, parts, (long long)C * Np, (long long)C * Np, nprob, 0);
    return LPVS_OK;
}

int ls_solve_accurate_multi(lpvs_ctx* c, const OpArgs& op, int Np, int zero_first, const double* d_Y, long long ldY, int C,
                            double* d_G, double lam, const std::function<int()>& regram, double* d_X, int* info) {
    cudaStream_t st = c->st;
    const int nb = Np / TB, ncc = op.ncc;
    const long long NN = (long long)Np * Np, N = op.N;
    const int nreal = 2 * ncc - zero_first;
    const double lam2 = lam * lam;
    int rc;
    for (int ch = 0; ch < C; ch++) info[ch] = 0;
    double* d_md = ws<double>(c, BUF_SUMS, 8);
    int* d_act = ws<int>(c, BUF_MC_ACT, (size_t)C);
    double* d_nrm = ws<double>(c, BUF_MC_NRM, (size_t)2 * C);
    double* d_g = ws<double>(c, BUF_MC_G, (size_t)2 * C * Np);  // g | tmp
    if (!d_md || !d_act || !d_nrm || !d_g) return fail(c, LPVS_E_NOMEM, "out of device memory (LS vectors of %d channels)", C);
    double* d_tmp = d_g + (long long)C * Np;
    std::vector<int> act((size_t)C);  // per channel: 1 still refining here, 0 done or handed on
    std::vector<int> route((size_t)C, 0);  // 0 primal refinement, 1 done (dual), 2 QR
    std::vector<double> h((size_t)2 * C), prev((size_t)C, 0.0);
    auto upload_act = [&]() -> int {
        LPVS_CU(c, cudaMemcpyAsync(d_act, act.data(), sizeof(int) * C, cudaMemcpyHostToDevice, st));
        return LPVS_OK;
    };
    auto read_norms = [&]() -> int {
        LPVS_CU(c, cudaMemcpyAsync(h.data(), d_nrm, sizeof(double) * 2 * C, cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaStreamSynchronize(st));
        return LPVS_OK;
    };
    GramArgs gb{};  // adjoint of the reference-rounded operator (as adjoint_apply)
    gb.t = op.t;
    gb.w_abs = 1;
    gb.s_end = N;
    gb.ncc = op.ncc;
    gb.nblk = nb;
    gb.tbl_ns = op.tbl_ns;
    gb.f = op.f;
    gb.gscale = 1.0;
    gb.bscale = op.dd;
    const unsigned gops = (unsigned)((N + 31) / 32), gch = (unsigned)((C + OPM_CW - 1) / OPM_CW);
    set_nt_smem(c);
    const size_t smem = (size_t)NT_STAGES * 2 * TILE_D * sizeof(double);
    const long long Nr = (N + TB - 1) / TB * TB;
    LPVS_CU(c, cudaMemsetAsync(d_X, 0, sizeof(double) * C * Np, st));

    // ---- 0. more functions than samples: the sample-space (dual) solve, the factor shared, the refinement per channel ----
    if (nreal >= N && lam > 0.0) {
        const int nbd = (int)(Nr / TB);
        double* d_A = ws<double>(c, BUF_LSQ_A, (size_t)Nr * Np);
        double* d_Gd = ws<double>(c, BUF_LSQ_G2, (size_t)std::max<long long>(Nr * Nr, NN));
        double* d_Xd = ws<double>(c, BUF_LSQ_LI, (size_t)std::max<long long>(Nr * Nr, NN));
        double* d_S = ws<double>(c, BUF_LSQ_Y, (size_t)std::max<long long>(Nr * Nr, NN));
        double* d_w = ws<double>(c, BUF_MC_W, (size_t)3 * C * Nr);  // w | r | dw
        double* Linv = ws<double>(c, BUF_LINV, (size_t)std::max(nbd, nb) * TB * TB);
        int* d_info = ws<int>(c, BUF_INFO, 1);
        if (!d_A || !d_Gd || !d_Xd || !d_S || !d_w || !Linv || !d_info)
            return fail(c, LPVS_E_NOMEM, "out of device memory (sample-space solve of %d channels)", C);
        double *d_r = d_w + (long long)C * Nr, *d_dw = d_w + 2LL * C * Nr;
        dim3 gm((unsigned)((Nr + 3) / 4), nb);
        k_materialize<<<gm, 256, 0, st>>>(op, d_A, Np, Nr);
        NtArgs t{};
        t.A = d_A; t.lda = Np;
        t.B = d_A; t.ldb = Np;
        t.C = d_Gd; t.ldc = Nr;
        t.mt = nbd; t.nt = nbd; t.mode = NT_SYRK;
        t.K = Np; t.Ksplit = Np;
        k_gemm_nt<<<nbd * (nbd + 1) / 2, NTHREADS, smem, st>>>(t);
        k_diag_dual<<<(unsigned)((Nr + 255) / 256), 256, 0, st>>>(d_Gd, Nr, N, lam2);
        c->launches += 3;
        CholArgs ca{};
        ca.G = d_Gd;
        ca.strideG = Nr * Nr;
        ca.Linv = Linv;
        ca.strideLinv = (long long)nbd * TB * TB;
        ca.info = d_info;
        ca.Np = (int)Nr;
        ca.nb = nbd;
        LPVS_CU(c, cudaMemsetAsync(ca.info, 0, sizeof(int), st));
        c->launches += potrf(ca, 1, c->sms, st, &c->la);
        k_pivot_range<<<1, 256, 0, st>>>(d_Gd, Nr, N, d_md + 4);
        c->launches++;
        int pinfo = 0;
        double pr[2] = {0.0, 0.0};
        LPVS_CU(c, cudaMemcpyAsync(&pinfo, ca.info, sizeof(int), cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaMemcpyAsync(pr, d_md + 4, sizeof pr, cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaStreamSynchronize(st));
        if (pinfo == 0 && pr[0] > 1e-10 * pr[1]) {  // ls_solve_dual's test: the factor can be refined against
            if ((rc = factor_inverse(c, d_Gd, Linv, (int)Nr, d_Xd, d_S))) return rc;
            LPVS_CU(c, cudaMemsetAsync(d_w, 0, sizeof(double) * 3 * C * Nr, st));
            for (int ch = 0; ch < C; ch++) act[ch] = 1;
            for (int step = 0; step < 6; step++) {
                if ((rc = upload_act())) return rc;
                k_op_apply_multi<<<dim3(gops, gch), 256, 0, st>>>(op, d_X, Np, d_Y, ldY, d_r, Nr, C);
                k_axpy_neg_multi<<<dim3((unsigned)((N + 255) / 256), C), 256, 0, st>>>(d_r, Nr, d_w, Nr, lam2, N);
                c->launches += 2;
                if ((rc = llt_solve_multi(c, d_Xd, (int)Nr, d_r, C, nullptr, d_dw, d_tmp))) return rc;  // Nr <= Np
                k_axpy_norms_multi<<<C, 1024, 0, st>>>(d_w, Nr, d_dw, Nr, (int)Nr, d_act, d_nrm);  // w += dw
                c->launches++;
                if ((rc = skinny_apply(c, d_A, Np, true, SK_FULL, Np, N, d_w, Nr, C, d_act, d_X, Np))) return rc;  // x = A'w
                if ((rc = read_norms())) return rc;
                bool any = false;
                for (int ch = 0; ch < C; ch++) {
                    if (!act[ch]) continue;
                    const double h0 = h[2 * ch], h1 = h[2 * ch + 1];
                    if (!(isfinite(h0) && isfinite(h1))) {  // NaN input: the caller's finite check reports the cause
                        act[ch] = 0;
                        route[ch] = 1;
                        continue;
                    }
                    const double rel = h1 > 0.0 ? sqrt(h0 / h1) : 0.0;
                    if (step > 0 && rel <= 1e-12) {
                        act[ch] = 0;
                        route[ch] = 1;
                        info[ch] = LPVS_INFO_DUAL;
                    } else if (step > 1 && rel > 0.25 * prev[ch]) {
                        act[ch] = 0;  // not contracting: the column-space path
                    } else {
                        prev[ch] = rel;
                        any = true;
                    }
                }
                if (!any) break;
            }
        }
    }
    int nprimal = 0;
    for (int ch = 0; ch < C; ch++) nprimal += route[ch] == 0;
    if (nprimal == 0) {
        LPVS_CU(c, cudaStreamSynchronize(st));
        return LPVS_OK;
    }

    // ---- 1. one factorisation for every channel: L L' = G~ + max(lam^2, n eps max diag) I (ls_solve_accurate's retries) ----
    int pinfo = 0;
    double mult = 1.0;
    double hmin[2] = {0.0, 0.0};
    for (int attempt = 0;; attempt++) {
        launch_max_diag(d_G, NN, Np, ncc, zero_first, d_md, 1, st);
        k_set_shift<<<1, 1, 0, st>>>(d_md, lam2, mult * (double)nreal * EPS);
        c->launches += 2;
        if ((rc = factor_solve(c, ncc, zero_first, Np, d_G, nullptr, 0, 0.0, 1, &pinfo, nullptr, 0.0, d_md + 1, attempt > 0)))
            return rc;
        k_min_pivot<<<1, 256, 0, st>>>(d_G, Np, ncc, zero_first, d_md + 4);
        c->launches++;
        LPVS_CU(c, cudaMemcpyAsync(&hmin[0], d_md + 4, sizeof(double), cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaMemcpyAsync(&hmin[1], d_md + 1, sizeof(double), cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaStreamSynchronize(st));
        if (pinfo == 0) break;
        if (attempt == 4 || !isfinite(mult)) {
            for (int ch = 0; ch < C; ch++) info[ch] = pinfo;
            return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown at internal pivot %d even with a %g n eps shift", pinfo, mult);
        }
        if (attempt > 0) mult *= 32.0;
        if ((rc = regram())) return rc;
    }
    const bool hopeless = hmin[0] < 8.0 * hmin[1];
    double* d_Li = ws<double>(c, BUF_LSQ_LI, (size_t)NN);
    double* d_G2 = ws<double>(c, BUF_LSQ_G2, (size_t)NN);
    double* d_R = ws<double>(c, BUF_MC_W, (size_t)C * (Nr + Np));  // residual [C][Mrows]
    double* Linv = ws<double>(c, BUF_LINV, (size_t)nb * TB * TB);
    if (!d_Li || !d_G2 || !d_R || !Linv) return fail(c, LPVS_E_NOMEM, "out of device memory (inverse factor, %d channels)", C);
    if ((rc = factor_inverse(c, d_G, Linv, Np, d_Li, d_G2))) return rc;  // X = L^-1 (d_G2: scratch until the SYRK)
    for (int ch = 0; ch < C; ch++) act[ch] = route[ch] == 0;
    if ((rc = upload_act())) return rc;

    // ---- 2. corrected semi-normal equations, C-wide; x0 = (L L')^-1 A'y ----
    if (!hopeless) {
        if ((rc = adjoint_apply_multi(c, gb, GRAM_DIRECT, Np, d_Y, ldY, C, d_g))) return rc;
        if ((rc = llt_solve_multi(c, d_Li, Np, d_g, C, d_act, d_X, d_tmp))) return rc;
        for (int step = 1; step <= 8; step++) {
            k_op_apply_multi<<<dim3(gops, gch), 256, 0, st>>>(op, d_X, Np, d_Y, ldY, d_R, N, C);
            c->launches++;
            if ((rc = adjoint_apply_multi(c, gb, GRAM_DIRECT, Np, d_R, N, C, d_g))) return rc;
            k_csne_rhs_multi<<<dim3((Np + 255) / 256, C), 256, 0, st>>>(d_g, d_X, lam2, Np, ncc, zero_first);
            c->launches++;
            if ((rc = llt_solve_multi(c, d_Li, Np, d_g, C, nullptr, d_g, d_tmp))) return rc;
            k_axpy_norms_multi<<<C, 1024, 0, st>>>(d_X, Np, d_g, Np, Np, d_act, d_nrm);
            c->launches++;
            if ((rc = read_norms())) return rc;
            bool any = false;
            for (int ch = 0; ch < C; ch++) {
                if (!act[ch]) continue;
                const double h0 = h[2 * ch], h1 = h[2 * ch + 1];
                act[ch] = 0;
                if (!(isfinite(h0) && isfinite(h1))) {
                    route[ch] = 2;
                    continue;
                }
                const double rel = h1 > 0.0 ? sqrt(h0 / h1) : 0.0;
                if (rel <= 1e-11) {
                    route[ch] = 1;  // converged: frozen
                } else if (rel > 0.05 * (step == 1 ? 1.0 : prev[ch])) {
                    route[ch] = 2;  // contraction too slow: the QR path
                } else {
                    prev[ch] = rel;
                    act[ch] = 1;
                    any = true;
                }
            }
            if (!any) break;
            if ((rc = upload_act())) return rc;
        }
        for (int ch = 0; ch < C; ch++)
            if (route[ch] == 0) route[ch] = 2;  // eight steps without converging
    } else {
        for (int ch = 0; ch < C; ch++)
            if (route[ch] == 0) route[ch] = 2;
    }
    int nqr = 0;
    for (int ch = 0; ch < C; ch++) {
        act[ch] = route[ch] == 2;
        nqr += act[ch];
    }
    if (nqr == 0) {
        LPVS_CU(c, cudaStreamSynchronize(st));
        return LPVS_OK;
    }
    if ((rc = upload_act())) return rc;
    for (int ch = 0; ch < C; ch++)
        if (act[ch]) info[ch] = LPVS_INFO_QR;

    // ---- 3. shifted CholeskyQR on the materialised regressor: the objects once, the solves for the marked channels ----
    const long long Mrows = Nr + Np;
    double* d_Yt = ws<double>(c, BUF_LSQ_Y, (size_t)NN);
    double* d_A = ws<double>(c, BUF_LSQ_A, (size_t)Nr * Np);
    double* d_Bt = ws<double>(c, BUF_LSQ_BT, (size_t)Np * Mrows);
    double* d_X2 = ws<double>(c, BUF_MC_X2, (size_t)NN);
    if (!d_Yt || !d_A || !d_Bt || !d_X2)
        return fail(c, LPVS_E_NOMEM, "out of device memory (QR path of a rank-deficient %d x %d problem)", (int)N, nreal);
    {
        dim3 grid(Np / 32, Np / 32);
        k_transpose_linv<<<grid, 256, 0, st>>>(d_Li, Np, ncc, zero_first, lam, d_Yt, d_Bt, Mrows, Nr);
        dim3 gm((unsigned)((Nr + 3) / 4), nb);
        k_materialize<<<gm, 256, 0, st>>>(op, d_A, Np, Nr);
        c->launches += 2;
    }
    NtArgs t1{};
    t1.A = d_Li; t1.lda = Np;
    t1.B = d_A; t1.ldb = Np;
    t1.C = d_Bt; t1.ldc = Mrows;
    t1.mt = nb; t1.nt = (int)(Nr / TB); t1.mode = NT_TRI;
    t1.K = Np; t1.Ksplit = 0;
    k_gemm_nt<<<t1.mt * t1.nt, NTHREADS, smem, st>>>(t1);
    NtArgs t2{};
    t2.A = d_Bt; t2.lda = Mrows;
    t2.B = d_Bt; t2.ldb = Mrows;
    t2.C = d_G2; t2.ldc = Np;
    t2.mt = nb; t2.nt = nb; t2.mode = NT_SYRK;
    t2.K = Mrows; t2.Ksplit = Nr;
    k_gemm_nt<<<nb * (nb + 1) / 2, NTHREADS, smem, st>>>(t2);
    c->launches += 2;
    if ((rc = factor_solve(c, ncc, zero_first, Np, d_G2, nullptr, 0, 0.0, 1, &pinfo))) return rc;
    LPVS_CU(c, cudaStreamSynchronize(st));
    if (pinfo) {  // once more with refined TRSM tiles
        k_gemm_nt<<<nb * (nb + 1) / 2, NTHREADS, smem, st>>>(t2);
        c->launches++;
        if ((rc = factor_solve(c, ncc, zero_first, Np, d_G2, nullptr, 0, 0.0, 1, &pinfo, nullptr, 0.0, nullptr, true)))
            return rc;
        LPVS_CU(c, cudaStreamSynchronize(st));
    }
    if (pinfo) {
        // last resort, shared: x = (G~ + shift I)^-1 A'y for the marked channels, LPVS_INFO_JITTER (as ls_solve_accurate)
        if ((rc = regram())) return rc;
        launch_max_diag(d_G, NN, Np, ncc, zero_first, d_md, 1, st);
        k_set_shift<<<1, 1, 0, st>>>(d_md, lam2, mult * (double)nreal * EPS);
        c->launches += 2;
        if ((rc = factor_solve(c, ncc, zero_first, Np, d_G, nullptr, 0, 0.0, 1, &pinfo, nullptr, 0.0, d_md + 1))) return rc;
        LPVS_CU(c, cudaStreamSynchronize(st));
        if (pinfo) {
            for (int ch = 0; ch < C; ch++) info[ch] = pinfo;
            return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown at internal pivot %d (rank-deficient problem, last resort)", pinfo);
        }
        if ((rc = factor_inverse(c, d_G, Linv, Np, d_Li, d_G2))) return rc;
        if ((rc = adjoint_apply_multi(c, gb, GRAM_DIRECT, Np, d_Y, ldY, C, d_g))) return rc;
        if ((rc = llt_solve_multi(c, d_Li, Np, d_g, C, d_act, d_X, d_tmp))) return rc;
        for (int ch = 0; ch < C; ch++)
            if (act[ch]) info[ch] = LPVS_INFO_JITTER;
        LPVS_CU(c, cudaStreamSynchronize(st));
        return LPVS_OK;
    }
    if ((rc = factor_inverse(c, d_G2, Linv, Np, d_X2, d_Yt))) return rc;  // L2^-1 (d_Yt: scratch, Y = X' is applied from X)
    // c = Q1'[y; 0], z = G2^-1 c, x = Y z
    if ((rc = skinny_apply(c, d_Bt, Mrows, false, SK_FULL, Np, N, d_Y, ldY, C, nullptr, d_g, Np))) return rc;
    if ((rc = llt_solve_multi(c, d_X2, Np, d_g, C, nullptr, d_g, d_tmp))) return rc;
    if ((rc = skinny_apply(c, d_Li, Np, true, SK_UPPER, Np, Np, d_g, Np, C, d_act, d_X, Np))) return rc;
    // refinement in the Q1 coordinates, per marked channel: dz = G2^-1 Q1'([y; 0] - [A; lam I] x), x += Y dz
    for (int step = 0; step < 2; step++) {
        LPVS_CU(c, cudaMemsetAsync(d_R, 0, sizeof(double) * C * Mrows, st));
        k_op_apply_multi<<<dim3(gops, gch), 256, 0, st>>>(op, d_X, Np, d_Y, ldY, d_R, Mrows, C);
        k_ridge_resid_multi<<<dim3((Np + 255) / 256, C), 256, 0, st>>>(d_R, Mrows, Nr, d_X, lam, Np, ncc, zero_first);
        c->launches += 2;
        if ((rc = skinny_apply(c, d_Bt, Mrows, false, SK_FULL, Np, Mrows, d_R, Mrows, C, nullptr, d_g, Np))) return rc;
        if ((rc = llt_solve_multi(c, d_X2, Np, d_g, C, nullptr, d_g, d_tmp))) return rc;
        if ((rc = skinny_apply(c, d_Li, Np, true, SK_UPPER, Np, Np, d_g, Np, C, nullptr, d_g, Np))) return rc;
        k_axpy_norms_multi<<<C, 1024, 0, st>>>(d_X, Np, d_g, Np, Np, d_act, d_nrm);
        c->launches++;
        if ((rc = read_norms())) return rc;
        bool any = false;
        for (int ch = 0; ch < C; ch++) {
            if (!act[ch]) continue;
            const double h0 = h[2 * ch], h1 = h[2 * ch + 1];
            // a second step only when the first one moved x by more than cond(G2) eps can explain
            if (!(isfinite(h0) && isfinite(h1)) || h0 <= 1e-16 * h1)
                act[ch] = 0;
            else
                any = true;
        }
        if (!any || step == 1) break;
        if ((rc = upload_act())) return rc;
    }
    LPVS_CU(c, cudaStreamSynchronize(st));
    return LPVS_OK;
}

}  // namespace lpvs
