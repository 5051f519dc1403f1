// Blocked FP64 Cholesky, triangular inverse and SPD inverse on 128x128 tiles.  See chol.cuh.
#include "chol.cuh"

#include <cooperative_groups.h>
namespace cg = cooperative_groups;

namespace lpvs {

namespace {

// ------------------------------------------------------------------------------------------------------------
// in-smem DMMA GEMM helper: C[MxN] = beta*C + alpha*A[MxK]*op(B); all operands in shared memory, row-major.
// BT: B is stored [N][K]; else [K][N].  M,N multiples of 8, K multiple of 4.  Tiles are spread over the warps.
// `lower`: skip 8x8 tiles strictly above the diagonal of C.
// ------------------------------------------------------------------------------------------------------------
template <bool BT>
__device__ __forceinline__ void smem_gemm(double* C, int ldc, const double* A, int lda, const double* B, int ldb,
                                          int M, int N, int K, double alpha, double beta, bool lower) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int tm = M >> 3, tn = N >> 3;
    const int r = lane >> 2, q = lane & 3;
    for (int tile = warp; tile < tm * tn; tile += nwarps) {
        int ti = tile / tn, tj = tile - ti * tn;
        if (lower && tj > ti) continue;
        double c0 = 0.0, c1 = 0.0, d0 = 0.0, d1 = 0.0;
        const double* pa = A + (8 * ti + r) * lda + q;
        const double* pb = BT ? (B + (8 * tj + r) * ldb + q) : (B + q * ldb + 8 * tj + r);
        int k0 = 0;
        for (; k0 + 8 <= K; k0 += 8) {  // two independent accumulator chains
            double a0 = pa[k0], a1 = pa[k0 + 4];
            double b0 = BT ? pb[k0] : pb[k0 * ldb];
            double b1 = BT ? pb[k0 + 4] : pb[(k0 + 4) * ldb];
            dmma884(c0, c1, a0, b0);
            dmma884(d0, d1, a1, b1);
        }
        for (; k0 < K; k0 += 4) {
            double a0 = pa[k0];
            double b0 = BT ? pb[k0] : pb[k0 * ldb];
            dmma884(c0, c1, a0, b0);
        }
        c0 += d0;
        c1 += d1;
        double* pc = C + (8 * ti + r) * ldc + 8 * tj + 2 * q;
        if (beta == 0.0) {
            pc[0] = alpha * c0;
            pc[1] = alpha * c1;
        } else {
            pc[0] = beta * pc[0] + alpha * c0;
            pc[1] = beta * pc[1] + alpha * c1;
        }
    }
}

constexpr int LDS = 132;  // 128x128 block stride (== 4 mod 16)
constexpr int PB = 16;    // inner panel width
constexpr int LDP = 20;   // stride of the 16x16 inverses
constexpr int LDH = 68;   // stride of the 64-row temp of the inverse phase

// smem layout of k_potf2: S[128*LDS] | T[64*LDH] | dinv[8][16*LDP] | LT[16*16] | colbuf[2*16]
constexpr int POTF2_SMEM_D = 128 * LDS + 64 * LDH + (TB / PB) * PB * LDP + PB * PB + 2 * PB;

// One warp, one 8-row tile row of C, up to NT adjacent 8x8 tiles (NT*2 independent DMMA chains):
//   C[8 x 8nt] (+)= alpha * A[8 x k0..k1) * op(B),  op(B)[k][n] = BT ? B[n*ldb + k] : B[k*ldb + n]
// A -> first row of the tile row, B -> first column of the first tile, C -> first element; k0, k1 multiples of 4.
template <bool BT, int NT>
__device__ __forceinline__ void warp_mma_row(double* C, int ldc, const double* A, int lda, const double* B, int ldb,
                                             int k0, int k1, int nt, double alpha, bool accumulate, int lane) {
    const int r = lane >> 2, q = lane & 3;
    double c[NT][2][2];
#pragma unroll
    for (int j = 0; j < NT; j++) c[j][0][0] = c[j][0][1] = c[j][1][0] = c[j][1][1] = 0.0;
    const double* pa = A + r * lda + q;
    const double* pb = BT ? (B + r * ldb + q) : (B + q * ldb + r);
    int k = k0;
    for (; k + 8 <= k1; k += 8) {
        const double a0 = pa[k], a1 = pa[k + 4];
#pragma unroll
        for (int j = 0; j < NT; j++)
            if (j < nt) {
                const double b0 = BT ? pb[8 * j * ldb + k] : pb[k * ldb + 8 * j];
                const double b1 = BT ? pb[8 * j * ldb + k + 4] : pb[(k + 4) * ldb + 8 * j];
                dmma884(c[j][0][0], c[j][0][1], a0, b0);
                dmma884(c[j][1][0], c[j][1][1], a1, b1);
            }
    }
    if (k < k1) {
        const double a0 = pa[k];
#pragma unroll
        for (int j = 0; j < NT; j++)
            if (j < nt) {
                const double b0 = BT ? pb[8 * j * ldb + k] : pb[k * ldb + 8 * j];
                dmma884(c[j][0][0], c[j][0][1], a0, b0);
            }
    }
    __syncwarp();  // in-place use (C aliases A): every lane has its operands before anyone stores
#pragma unroll
    for (int j = 0; j < NT; j++)
        if (j < nt) {
            double2* pc = reinterpret_cast<double2*>(C + r * ldc + 8 * j + 2 * q);
            double2 v = make_double2(alpha * (c[j][0][0] + c[j][1][0]), alpha * (c[j][0][1] + c[j][1][1]));
            if (accumulate) {
                const double2 o = *pc;
                v.x += o.x;
                v.y += o.y;
            }
            *pc = v;
        }
}

// One warp factorises a 16x16 SPD block AND inverts the factor, in lockstep: lanes 0-15 own row (lane) of the block, lanes
// 16-31 own column (lane - 16) of X = L^-1.  Column c of the factor is broadcast UNSCALED through shared memory (double-
// buffered, one __syncwarp per column) while the pivot travels by shuffle; the scaling by rsqrt(pivot) is applied to the
// multiplier instead of to the column (an LDL'-style update), so the critical path per column is pivot -> rsqrt -> two
// multiplies -> one FMA.  The inverse needs exactly that broadcast column: its running sums s[i] = sum_{k<=c} L[i][k] x[k]
// advance by the same FMA with the multiplier rsqrt(pivot) * x[c], and x[c] = -s[c] rsqrt(pivot) is ready when column c is.
// Both halves therefore execute ONE instruction stream.  Measured (tools/potf2_probe.cu): 5.9 K cycles per panel, the same as
// the two-loop version -- the panel is a chain of dependent FP64 operations at ~365 cycles per column, not issue-bound.  A
// reciprocal-only chain (MUFU.RCP64H seed + two Newton steps for the multiplier, rsqrt taken once after the loop) was also
// measured and is SLOWER (7.1 K cycles): CUDA's rsqrt is the shorter dependent sequence on this pipe.
__device__ __forceinline__ void warp_potf2_inv(double* D, int ldd, double* Di, int ldi, double* colbuf, int lane,
                                               int* info, int pivot_base, double tol) {
    const unsigned full = 0xffffffffu;
    const int row = lane & (PB - 1);
    const bool inv = lane >= PB;
    double a[PB];  // factor lanes: A[row][.] -> L[row][.]; inverse lanes: running sums -> X[.][row]
#pragma unroll
    for (int c = 0; c < PB; c++) a[c] = (!inv && c <= row) ? D[row * ldd + c] : 0.0;
#pragma unroll
    for (int c = 0; c < PB; c++) {
        double* cb = colbuf + (c & 1) * PB;
        if (!inv) cb[row] = a[c];
        double piv = __shfl_sync(full, a[c], c);
        if (!(piv > tol) || !isfinite(piv)) {
            if (lane == 0) atomicCAS(info, 0, pivot_base + c + 1);
            piv = (fabs(piv) > 0.0 && isfinite(piv)) ? fabs(piv) : 1.0;
        }
        const double ri = rsqrt(piv);
        double keep, mult;
        if (!inv) {
            keep = (row == c) ? piv * ri : a[c] * ri;  // L[row][c]
            mult = -(keep * ri);                        // -a[row][c] / pivot
        } else {
            keep = (c == row) ? ri : ((c > row) ? -a[c] * ri : 0.0);  // X[c][row]
            mult = ri * keep;
        }
        a[c] = keep;
        __syncwarp();
#pragma unroll
        for (int kk = (c + 1) / 2; kk < PB / 2; kk++) {
            const double2 v = reinterpret_cast<const double2*>(cb)[kk];
            if (2 * kk > c) a[2 * kk] = fma(mult, v.x, a[2 * kk]);
            a[2 * kk + 1] = fma(mult, v.y, a[2 * kk + 1]);
        }
    }
    if (!inv) {
#pragma unroll
        for (int c = 0; c < PB; c++)
            if (c <= row) D[row * ldd + c] = a[c];
    } else {
#pragma unroll
        for (int c = 0; c < PB; c++) Di[c * ldi + row] = a[c];
    }
}

#ifdef LPVS_POTF2_TRACE  // tools/potf2_probe.cu: clock stamps of CTA 0
__device__ long long* g_potf2_trace;
#define POTF2_TR(slot) if (blockIdx.x == 0 && threadIdx.x == 0) g_potf2_trace[slot] = clock64();
#else
#define POTF2_TR(slot)
#endif

// 128x128 diagonal block: L_kk (in place in G) and its inverse (Linv), one CTA per problem.
__global__ void __launch_bounds__(NTHREADS, 1) k_potf2(const __grid_constant__ CholArgs a, int k) {
    extern __shared__ __align__(16) double sm[];
    double* S = sm;
    double* T = sm + 128 * LDS;
    double* Dinv = T + 64 * LDH;
    double* colbuf = Dinv + (TB / PB) * PB * LDP + PB * PB;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int prob = blockIdx.x;
    double* Gd = a.G + (long long)prob * a.strideG + ((long long)k * TB) * a.Np + (long long)k * TB;
    const double tol = a.maxdiag ? a.maxdiag[prob] * a.tol_scale : 0.0;
    POTF2_TR(0)

    // lower triangle of the diagonal block: all 16-byte pieces in flight at once (cp.async); zeros above
    for (int idx = tid; idx < TB * TB / 2; idx += NTHREADS) {
        const int r = idx >> 6, c = (idx & 63) * 2;
        if (c <= r)
            cp_async16(S + r * LDS + c, Gd + (long long)r * a.Np + c);
        else
            *reinterpret_cast<double2*>(S + r * LDS + c) = make_double2(0.0, 0.0);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    POTF2_TR(1)

    // Left-looking over 16-column panels with look-ahead: while warp 0 runs the serial 16x16 factor + inverse of panel p
    // (5.7 K cycles, tools/potf2_probe.cu), warps 1-7 already apply the finished columns [0, 16p) to panel p+1, so after
    // the panel's TRSM only its own rank-16 contribution to panel p+1 is left.  Every tile is read-modify-written a few
    // times with long DMMA chains instead of once per panel with chains of 4.
    for (int p = 0; p < TB / PB; p++) {
        const int j0 = p * PB;
        double* Di = Dinv + p * PB * LDP;
        const int nt = (TB - j0 - PB) >> 3;  // 8-row tiles below the panel's diagonal block
        if (warp == 0) {
            warp_potf2_inv(S + j0 * LDS + j0, LDS, Di, LDP, colbuf, lane, &a.info[prob], k * TB + j0, tol);
        } else if (nt > 0 && j0 > 0 && warp != 4) {
            // panel p+1 (columns j0+16 .. j0+31, rows >= j0+16) -= L[rows, 0:j0) * L[j0+16 .. j0+31, 0:j0)'
            // Warp 4 shares warp 0's SM sub-partition, i.e. its FP64 pipe: every DMMA it issued here could hold one of the
            // dependent FP64 operations of warp 0's pivot chain back by up to 16 cycles, so it sits this phase out
            // (5.95 K -> 5.85 K cycles per panel, tools/potf2_probe.cu).
            const double* Brow = S + (j0 + PB) * LDS;
            for (int ti = warp < 4 ? warp - 1 : warp - 2; ti < nt; ti += NTHREADS / 32 - 2)
                warp_mma_row<true, 2>(S + (j0 + PB + 8 * ti) * LDS + j0 + PB, LDS, S + (j0 + PB + 8 * ti) * LDS, LDS, Brow,
                                      LDS, 0, j0, 2, -1.0, true, lane);
        }
        __syncthreads();
        POTF2_TR(2 + 2 * p)
        if (nt > 0) {
            double* P = S + (j0 + PB) * LDS + j0;  // panel below the diagonal block
            // P <- P * Dinv' in place (a warp owns whole tile rows)
            for (int ti = warp; ti < nt; ti += NTHREADS / 32)
                warp_mma_row<true, 2>(P + 8 * ti * LDS, LDS, P + 8 * ti * LDS, LDS, Di, LDP, 0, PB, 2, 1.0, false, lane);
            __syncthreads();
            // panel p+1 -= P P[0:16]'  (this panel's own contribution)
            for (int ti = warp; ti < nt; ti += NTHREADS / 32)
                warp_mma_row<true, 2>(S + (j0 + PB + 8 * ti) * LDS + j0 + PB, LDS, P + 8 * ti * LDS, LDS, P, LDS, 0, PB, 2,
                                      -1.0, true, lane);
            __syncthreads();
        }
        POTF2_TR(3 + 2 * p)
    }

    // write L_kk back (strictly-upper part of the block zeroed)
    for (int idx = tid; idx < TB * TB / 2; idx += NTHREADS) {
        const int r = idx >> 6, c = (idx & 63) * 2;
        double2 v = *reinterpret_cast<const double2*>(S + r * LDS + c);
        if (c > r) v.x = 0.0;
        if (c + 1 > r) v.y = 0.0;
        *reinterpret_cast<double2*>(Gd + (long long)r * a.Np + c) = v;
    }
    __syncthreads();
    POTF2_TR(18)

    // in-place inverse: diagonal 16x16 blocks first, then recursive doubling X21 = -X22 (L21 X11), all pairs of a
    // level at once, zero blocks of the triangular factors skipped
    for (int idx = tid; idx < (TB / PB) * PB * PB; idx += NTHREADS) {
        int p = idx >> 8, r = (idx >> 4) & 15, c = idx & 15;
        S[(p * PB + r) * LDS + p * PB + c] = (c <= r) ? Dinv[p * PB * LDP + r * LDP + c] : 0.0;
    }
    __syncthreads();
    for (int h = PB; h < TB; h <<= 1) {
        const int ht = h >> 3;                 // tiles per side of a sub-block
        const int ng = (ht + 3) >> 2;          // tile groups per tile row
        const int npair = TB / (2 * h);
        const int nunits = npair * ht * ng;
        // T_pair = L21 * X11  (X11 lower triangular: k >= first column of the group)
        for (int u = warp; u < nunits; u += NTHREADS / 32) {
            const int pr = u / (ht * ng), rem = u - pr * ht * ng, ti = rem / ng, g = (rem - ti * ng) * 4;
            const int o = pr * 2 * h;
            warp_mma_row<false, 4>(T + (pr * h + 8 * ti) * LDH + 8 * g, LDH, S + (o + h + 8 * ti) * LDS + o, LDS,
                                   S + o * LDS + o + 8 * g, LDS, 8 * g, h, min(4, ht - g), 1.0, false, lane);
        }
        __syncthreads();
        // X21 = -X22 * T_pair  (X22 lower triangular: k <= last row of the tile row)
        for (int u = warp; u < nunits; u += NTHREADS / 32) {
            const int pr = u / (ht * ng), rem = u - pr * ht * ng, ti = rem / ng, g = (rem - ti * ng) * 4;
            const int o = pr * 2 * h;
            warp_mma_row<false, 4>(S + (o + h + 8 * ti) * LDS + o + 8 * g, LDS, S + (o + h + 8 * ti) * LDS + o + h, LDS,
                                   T + pr * h * LDH + 8 * g, LDH, 0, 8 * (ti + 1), min(4, ht - g), -1.0, false, lane);
        }
        __syncthreads();
    }
    POTF2_TR(19)
    if (a.rhs) {
        // fused forward substitution: y_k = Linv_kk r_k (r_k already carries -sum_{j<k} L_kj y_j from the TRSM tiles)
        double* rk = a.rhs + (long long)prob * a.strideRhs + (long long)k * TB;
        for (int q = tid; q < 2 * TB; q += NTHREADS) T[q] = (q >> 7) < a.nrhs ? __ldcg(rk + (long long)(q >> 7) * a.Np + (q & 127)) : 0.0;
        __syncthreads();
        for (int rr = warp; rr < TB; rr += NTHREADS / 32) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int c = lane + 32 * q;
                const double l = c <= rr ? S[rr * LDS + c] : 0.0;
                s0 = fma(l, T[c], s0);
                s1 = fma(l, T[TB + c], s1);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            }
            if (lane == 0) {
                rk[rr] = s0;
                if (a.nrhs > 1) rk[a.Np + rr] = s1;
            }
        }
    }
    double* Li = a.Linv + (long long)prob * a.strideLinv + (long long)k * TB * TB;
    for (int idx = tid; idx < TB * TB / 2; idx += NTHREADS) {
        const int r = idx >> 6, c = (idx & 63) * 2;
        double2 v = *reinterpret_cast<const double2*>(S + r * LDS + c);
        if (c > r) v.x = 0.0;
        if (c + 1 > r) v.y = 0.0;
        *reinterpret_cast<double2*>(Li + r * TB + c) = v;
    }
    POTF2_TR(20)
}

// ------------------------------------------------------------------------------------------------------------
// global-memory NT GEMM tile: acc += A[128 x K] * B[128 x K]' with cp.async double buffering
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NTHREADS, 1) k_gemm(const __grid_constant__ CholArgs a, int mode, int k) {
    extern __shared__ __align__(16) double sm[];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int wm = w & 3, wn = w >> 2;
    const int prob = blockIdx.y;
    const int t = blockIdx.x;
    const long long Np = a.Np;
    double* G = a.G + (long long)prob * a.strideG;
    double* Y = a.Y ? a.Y + (long long)prob * a.strideY : nullptr;
    const double* Linv = a.Linv + (long long)prob * a.strideLinv;

    const double *A, *B;
    double* C;
    long long lda, ldb, ldc = Np;
    int K;
    double alpha, beta;
    switch (mode) {
        case GM_TRSM_RES: {
            int i = k + 1 + t;
            A = G + (long long)i * TB * Np + (long long)k * TB; lda = Np;
            B = G + (long long)k * TB * Np + (long long)k * TB; ldb = Np;  // L_kk (zeros above its diagonal)
            C = a.trsm_scratch + (long long)t * TB * TB; ldc = TB;
            K = TB; alpha = -1.0; beta = 1.0;
        } break;
        case GM_TRSM_FIX: {
            int i = k + 1 + t;
            A = a.trsm_scratch + (long long)t * TB * TB; lda = TB;
            B = Linv + (long long)k * TB * TB; ldb = TB;
            C = G + (long long)i * TB * Np + (long long)k * TB;
            K = TB; alpha = 1.0; beta = 1.0;
        } break;
        case GM_TRSM: {
            int i = k + 1 + t;
            A = G + (long long)i * TB * Np + (long long)k * TB; lda = Np;
            B = Linv + (long long)k * TB * TB; ldb = TB;
            C = G + (long long)i * TB * Np + (long long)k * TB;
            K = TB; alpha = 1.0; beta = 0.0;
        } break;
        case GM_SYRK_RIGHT: {
            int ii, jj;
            tile_ij(t, ii, jj);
            int i = k + 1 + ii, j = k + 1 + jj;
            A = G + (long long)i * TB * Np + (long long)k * TB; lda = Np;
            B = G + (long long)j * TB * Np + (long long)k * TB; ldb = Np;
            C = G + (long long)i * TB * Np + (long long)j * TB;
            K = TB; alpha = -1.0; beta = 1.0;
        } break;
        case GM_SYRK_COL: {
            int i = k + 1 + t, j = k + 1;
            A = G + (long long)i * TB * Np + (long long)k * TB; lda = Np;
            B = G + (long long)j * TB * Np + (long long)k * TB; ldb = Np;
            C = G + (long long)i * TB * Np + (long long)j * TB;
            K = TB; alpha = -1.0; beta = 1.0;
        } break;
        case GM_SYRK_REST: {
            int ii, jj;
            tile_ij(t, ii, jj);
            int i = k + 2 + ii, j = k + 2 + jj;
            A = G + (long long)i * TB * Np + (long long)k * TB; lda = Np;
            B = G + (long long)j * TB * Np + (long long)k * TB; ldb = Np;
            C = G + (long long)i * TB * Np + (long long)j * TB;
            K = TB; alpha = -1.0; beta = 1.0;
        } break;
        case GM_SYRK_LEFT: {
            int i = k + t;
            A = G + (long long)i * TB * Np; lda = Np;
            B = G + (long long)k * TB * Np; ldb = Np;
            C = G + (long long)i * TB * Np + (long long)k * TB;
            K = k * TB; alpha = -1.0; beta = 1.0;
        } break;
        case GM_TRTRI_A: {
            int kb = t;  // kb < k (k plays the role of block column i)
            A = Y + (long long)kb * TB * Np + (long long)kb * TB; lda = Np;
            B = G + (long long)k * TB * Np + (long long)kb * TB; ldb = Np;
            C = Y + (long long)kb * TB * Np + (long long)k * TB;
            K = (k - kb) * TB; alpha = 1.0; beta = 0.0;
        } break;
        case GM_TRTRI_B: {
            int kb = t;
            A = Y + (long long)kb * TB * Np + (long long)k * TB; lda = Np;
            B = Linv + (long long)k * TB * TB; ldb = TB;
            C = Y + (long long)kb * TB * Np + (long long)k * TB;
            K = TB; alpha = -1.0; beta = 0.0;
        } break;
        default: {  // GM_LAUUM
            int ia, ib;
            tile_ij(t, ia, ib);
            A = Y + (long long)ia * TB * Np + (long long)ia * TB; lda = Np;
            B = Y + (long long)ib * TB * Np + (long long)ia * TB; ldb = Np;
            C = G + (long long)ia * TB * Np + (long long)ib * TB;
            K = (a.nb - ia) * TB; alpha = 1.0; beta = 0.0;
        } break;
    }

    double acc[4][8][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

    __shared__ double ysm[2][TB];       // y_k of the fused forward substitution (TRSM only)
    __shared__ double yred[2][2][TB];   // [wn][rhs][row]
    const bool fwd = mode == GM_TRSM && a.rhs != nullptr;
    if (fwd) {
        const double* yk = a.rhs + (long long)prob * a.strideRhs + (long long)k * TB;
        ysm[tid >> 7][tid & 127] = (tid >> 7) < a.nrhs ? __ldcg(yk + (long long)(tid >> 7) * Np + (tid & 127)) : 0.0;
    }
    const int nchunks = K / KC;
    double* st0 = sm;
    double* st1 = sm + 2 * TILE_D;
    if (nchunks > 0) {
        load_tile_async(st0, A, lda, tid);
        load_tile_async(st0 + TILE_D, B, ldb, tid);
    }
    cp_async_commit();
    const int fragA = (32 * wm + (lane >> 2)) * LDT + (lane & 3);
    const int fragB = (64 * wn + (lane >> 2)) * LDT + (lane & 3);
    for (int c = 0; c < nchunks; c++) {
        double* cur = (c & 1) ? st1 : st0;
        double* nxt = (c & 1) ? st0 : st1;
        if (c + 1 < nchunks) {
            load_tile_async(nxt, A + (long long)(c + 1) * KC, lda, tid);
            load_tile_async(nxt + TILE_D, B + (long long)(c + 1) * KC, ldb, tid);
        }
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        const double* pa = cur + fragA;
        const double* pb = cur + TILE_D + fragB;
#pragma unroll
        for (int kk = 0; kk < KC / 4; kk++) mma_step(pa, pb, kk, acc);
        __syncthreads();
    }
    cp_async_wait<0>();

#pragma unroll
    for (int i = 0; i < 4; i++) {
        int row = 32 * wm + 8 * i + (lane >> 2);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            int col = 64 * wn + 8 * j + 2 * (lane & 3);
            double2* pc = reinterpret_cast<double2*>(C + (long long)row * ldc + col);
            double2 v = make_double2(alpha * acc[i][j][0], alpha * acc[i][j][1]);
            if (beta != 0.0) {
                double2 o = *pc;
                v.x += beta * o.x;
                v.y += beta * o.y;
            }
            *pc = v;
        }
    }
    if (fwd) {
        // r_i -= L_ik y_k for this tile's 128 rows (this CTA is the only writer of r_i in this launch)
#pragma unroll
        for (int i = 0; i < 4; i++) {
            double p0 = 0.0, p1 = 0.0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int col = 64 * wn + 8 * j + 2 * (lane & 3);
                p0 = fma(acc[i][j][0], ysm[0][col], fma(acc[i][j][1], ysm[0][col + 1], p0));
                p1 = fma(acc[i][j][0], ysm[1][col], fma(acc[i][j][1], ysm[1][col + 1], p1));
            }
            p0 += __shfl_xor_sync(0xffffffffu, p0, 1);
            p0 += __shfl_xor_sync(0xffffffffu, p0, 2);
            p1 += __shfl_xor_sync(0xffffffffu, p1, 1);
            p1 += __shfl_xor_sync(0xffffffffu, p1, 2);
            if ((lane & 3) == 0) {
                const int row = 32 * wm + 8 * i + (lane >> 2);
                yred[wn][0][row] = p0;
                yred[wn][1][row] = p1;
            }
        }
        __syncthreads();
        const int v = tid >> 7, row = tid & 127;
        if (v < a.nrhs) {
            double* ri = a.rhs + (long long)prob * a.strideRhs + (long long)v * Np + (long long)(k + 1 + t) * TB + row;
            *ri -= yred[0][v][row] + yred[1][v][row];
        }
    }
}

__global__ void k_diag_prepare(double* G, long long strideG, int Np, int ncc, int zero_first,
                               const double* __restrict__ ridge_dev, double ridge) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Np) return;
    int prob = blockIdx.y;
    double* g = G + (long long)prob * strideG + (long long)i * Np + i;
    double rg = ridge_dev ? ridge_dev[prob] : ridge;
    *g = is_dummy_col(i, ncc, zero_first) ? 1.0 : (*g + rg);
}

__global__ void k_max_diag(const double* __restrict__ G, long long strideG, int Np, int ncc, int zero_first,
                           double* out) {
    __shared__ double red[256];
    int prob = blockIdx.x;
    const double* g = G + (long long)prob * strideG;
    double m = 0.0;
    for (int i = threadIdx.x; i < Np; i += blockDim.x)
        if (!is_dummy_col(i, ncc, zero_first)) m = fmax(m, fabs(g[(long long)i * Np + i]));
    red[threadIdx.x] = m;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] = fmax(red[threadIdx.x], red[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) out[prob] = red[0];
}

__global__ void k_init_y(const __grid_constant__ CholArgs a) {
    // Y_kk = Linv_kk'
    int kb = blockIdx.x, prob = blockIdx.y;
    const double* Li = a.Linv + (long long)prob * a.strideLinv + (long long)kb * TB * TB;
    double* Yd = a.Y + (long long)prob * a.strideY + (long long)kb * TB * a.Np + (long long)kb * TB;
    __shared__ double tile[32][33];
    for (int br = 0; br < TB; br += 32)
        for (int bc = 0; bc < TB; bc += 32) {
            int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 256 threads: 8 rows at a time
            for (int r = ty; r < 32; r += 8) tile[r][tx] = Li[(br + r) * TB + bc + tx];
            __syncthreads();
            for (int r = ty; r < 32; r += 8) Yd[(long long)(bc + r) * a.Np + br + tx] = tile[tx][r];
            __syncthreads();
        }
}

__global__ void k_symmetrize(double* G, long long strideG, int Np) {
    // copy lower 32x32 tiles to upper
    int bi = blockIdx.x, bj = blockIdx.y, prob = blockIdx.z;
    if (bj >= bi) return;
    double* g = G + (long long)prob * strideG;
    __shared__ double tile[32][33];
    int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) tile[r][tx] = g[(long long)(bi * 32 + r) * Np + bj * 32 + tx];
    __syncthreads();
    for (int r = ty; r < 32; r += 8) g[(long long)(bj * 32 + r) * Np + bi * 32 + tx] = tile[tx][r];
}

// ------------------------------------------------------------------------------------------------------------
// blocked TRSV with the pre-inverted diagonal blocks; one CTA per problem, up to 2 right-hand sides
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(NTHREADS, 1) k_trsv(const __grid_constant__ CholArgs a, double* Bm,
                                                      long long strideB, int nrhs, int fwd_done) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int prob = blockIdx.x;
    const long long Np = a.Np;
    const double* L = a.G + (long long)prob * a.strideG;
    const double* Linv = a.Linv + (long long)prob * a.strideLinv;
    double* b = Bm + (long long)prob * strideB;  // [nrhs][Np], solved in place
    __shared__ double rbuf[2][TB];
    __shared__ double part[2][2][TB];

    // forward: L y = b
    for (int kb = fwd_done ? a.nb : 0; kb < a.nb; kb++) {
        for (int rr = warp; rr < TB; rr += 8) {
            const double* row = L + (long long)(kb * TB + rr) * Np;
            double s0 = 0.0, s1 = 0.0;
            for (int c = lane; c < kb * TB; c += 32) {
                double l = row[c];
                s0 += l * __ldcg(b + c);
                if (nrhs > 1) s1 += l * __ldcg(b + Np + c);
            }
            s0 = warp_sum(s0);
            s1 = warp_sum(s1);
            if (lane == 0) {
                rbuf[0][rr] = __ldcg(b + kb * TB + rr) - s0;
                if (nrhs > 1) rbuf[1][rr] = __ldcg(b + Np + kb * TB + rr) - s1;
            }
        }
        __syncthreads();
        const double* Li = Linv + (long long)kb * TB * TB;
        for (int rr = warp; rr < TB; rr += 8) {
            double s0 = 0.0, s1 = 0.0;
            for (int c = lane; c <= rr; c += 32) {
                double l = Li[rr * TB + c];
                s0 += l * rbuf[0][c];
                if (nrhs > 1) s1 += l * rbuf[1][c];
            }
            s0 = warp_sum(s0);
            s1 = warp_sum(s1);
            if (lane == 0) {
                b[kb * TB + rr] = s0;
                if (nrhs > 1) b[Np + kb * TB + rr] = s1;
            }
        }
        __syncthreads();
    }
    // backward: L' x = y
    const int c = tid & 127, h = tid >> 7;
    for (int kb = a.nb - 1; kb >= 0; kb--) {
        double s0 = 0.0, s1 = 0.0;
        for (long long r = (long long)(kb + 1) * TB + h; r < Np; r += 2) {
            double l = L[r * Np + kb * TB + c];
            s0 += l * __ldcg(b + r);
            if (nrhs > 1) s1 += l * __ldcg(b + Np + r);
        }
        part[0][h][c] = s0;
        part[1][h][c] = s1;
        __syncthreads();
        if (h == 0) {
            rbuf[0][c] = __ldcg(b + kb * TB + c) - (part[0][0][c] + part[0][1][c]);
            if (nrhs > 1) rbuf[1][c] = __ldcg(b + Np + kb * TB + c) - (part[1][0][c] + part[1][1][c]);
        }
        __syncthreads();
        const double* Li = Linv + (long long)kb * TB * TB;
        s0 = 0.0;
        s1 = 0.0;
        for (int m = c + h; m < TB; m += 2) {
            double l = Li[m * TB + c];
            s0 += l * rbuf[0][m];
            if (nrhs > 1) s1 += l * rbuf[1][m];
        }
        part[0][h][c] = s0;
        part[1][h][c] = s1;
        __syncthreads();
        if (h == 0) {
            b[kb * TB + c] = part[0][0][c] + part[0][1][c];
            if (nrhs > 1) b[Np + kb * TB + c] = part[1][0][c] + part[1][1][c];
        }
        __syncthreads();
    }
}

// Backward substitution only (L' x = y), one CTA per problem, for the batched path whose forward substitution was
// fused into the factorisation.  x lives in shared memory; thread (c, h) walks every TRSV_H-th row of column c of the
// block column below the diagonal block (coalesced 1 KB row pieces, 8 independent loads in flight per thread).
constexpr int TRSV_T = 512, TRSV_H = TRSV_T / TB;
__global__ void __launch_bounds__(TRSV_T, 2) k_trsv_bwd(const __grid_constant__ CholArgs a, double* Bm, long long strideB,
                                                        int nrhs) {
    extern __shared__ __align__(16) double xs[];  // [2][Np]
    __shared__ double part[2][TRSV_H][TB];
    __shared__ double rbuf[2][TB];
    const int tid = threadIdx.x, c = tid & 127, h = tid >> 7;
    const int prob = blockIdx.x;
    const int Np = a.Np;
    const double* L = a.G + (long long)prob * a.strideG;
    const double* Linv = a.Linv + (long long)prob * a.strideLinv;
    double* b = Bm + (long long)prob * strideB;
    if (__ldcg(a.info + prob) != 0) return;  // broken factorisation: nothing to solve
    for (int q = tid; q < 2 * Np; q += TRSV_T) xs[q] = (q / Np) < nrhs ? __ldcg(b + q) : 0.0;
    __syncthreads();
    for (int kb = a.nb - 1; kb >= 0; kb--) {
        double s0 = 0.0, s1 = 0.0;
        const double* col = L + (long long)kb * TB + c;
        int r = (kb + 1) * TB + h;
        for (; r + 7 * TRSV_H < Np; r += 8 * TRSV_H) {
            double l[8];
#pragma unroll
            for (int q = 0; q < 8; q++) l[q] = __ldcs(col + (long long)(r + q * TRSV_H) * Np);
#pragma unroll
            for (int q = 0; q < 8; q++) {
                s0 = fma(l[q], xs[r + q * TRSV_H], s0);
                s1 = fma(l[q], xs[Np + r + q * TRSV_H], s1);
            }
        }
        for (; r < Np; r += TRSV_H) {
            const double l = __ldcs(col + (long long)r * Np);
            s0 = fma(l, xs[r], s0);
            s1 = fma(l, xs[Np + r], s1);
        }
        part[0][h][c] = s0;
        part[1][h][c] = s1;
        __syncthreads();
        if (h < 2) {  // h = rhs here
            double t = 0.0;
#pragma unroll
            for (int q = 0; q < TRSV_H; q++) t += part[h][q][c];
            rbuf[h][c] = xs[h * Np + kb * TB + c] - t;
        }
        __syncthreads();
        // x_k = Linv_kk' rbuf: column c of Linv', rows m >= c
        const double* Li = Linv + (long long)kb * TB * TB;
        s0 = 0.0;
        s1 = 0.0;
        for (int m = c + h; m < TB; m += TRSV_H) {
            const double l = Li[m * TB + c];
            s0 = fma(l, rbuf[0][m], s0);
            s1 = fma(l, rbuf[1][m], s1);
        }
        part[0][h][c] = s0;
        part[1][h][c] = s1;
        __syncthreads();
        if (h < 2) {
            double t = 0.0;
#pragma unroll
            for (int q = 0; q < TRSV_H; q++) t += part[h][q][c];
            xs[h * Np + kb * TB + c] = t;
            if (h < nrhs) b[(long long)h * Np + kb * TB + c] = t;
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------------
// multi-CTA blocked TRSV for ONE large problem (cooperative launch, grid = nb CTAs, CTA i owns row block i).
// Forward:  y_k = Linv_k r_k, publish, then every CTA i > k does r_i -= L[i,k] y_k.   One grid barrier per block.
// Backward: x_k = Linv_k' r_k, publish, then every CTA i < k does r_i -= L[k,i]' x_k.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NTHREADS, 1) k_trsv_big(const __grid_constant__ CholArgs a, double* b, int nrhs,
                                                          int fwd_done) {
    cg::grid_group grid = cg::this_grid();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int i = blockIdx.x;
    const long long Np = a.Np;
    const double* L = a.G;
    if (__ldcg(a.info) != 0) return;  // broken factorisation (set before this launch): every CTA leaves, the host retries
    __shared__ double r[2][TB];     // this CTA's running right-hand side block
    __shared__ double yk[2][TB];    // the published solution block of the current step
    __shared__ double part[2][2][TB];
    for (int q = tid; q < 2 * TB; q += NTHREADS) {
        int rh = q >> 7, c = q & 127;
        r[rh][c] = rh < nrhs ? b[(long long)rh * Np + i * TB + c] : 0.0;
    }
    __syncthreads();
    // ---- forward ---- (skipped when the factorisation already produced y, see CholArgs::rhs)
    for (int k = fwd_done ? a.nb : 0; k < a.nb; k++) {
        if (i == k) {
            const double* Li = a.Linv + (long long)k * TB * TB;
            for (int rr = warp; rr < TB; rr += 8) {
                double s0 = 0.0, s1 = 0.0;
                for (int c = lane; c <= rr; c += 32) {
                    double l = Li[rr * TB + c];
                    s0 = fma(l, r[0][c], s0);
                    s1 = fma(l, r[1][c], s1);
                }
                s0 = warp_sum(s0);
                s1 = warp_sum(s1);
                if (lane == 0) {
                    b[k * TB + rr] = s0;
                    if (nrhs > 1) b[Np + k * TB + rr] = s1;
                }
            }
        }
        grid.sync();
        if (i > k) {
            for (int q = tid; q < 2 * TB; q += NTHREADS) {
                int rh = q >> 7, c = q & 127;
                yk[rh][c] = rh < nrhs ? __ldcg(b + (long long)rh * Np + k * TB + c) : 0.0;
            }
            __syncthreads();
            const double* T = L + (long long)i * TB * Np + (long long)k * TB;
            for (int rr = warp; rr < TB; rr += 8) {
                const double* row = T + (long long)rr * Np;
                double s0 = 0.0, s1 = 0.0;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    double l = row[lane + 32 * q];
                    s0 = fma(l, yk[0][lane + 32 * q], s0);
                    s1 = fma(l, yk[1][lane + 32 * q], s1);
                }
                s0 = warp_sum(s0);
                s1 = warp_sum(s1);
                if (lane == 0) {
                    r[0][rr] -= s0;
                    r[1][rr] -= s1;
                }
            }
            __syncthreads();
        }
    }
    // r of CTA i is now stale; reload y_i as the backward right-hand side
    grid.sync();
    for (int q = tid; q < 2 * TB; q += NTHREADS) {
        int rh = q >> 7, c = q & 127;
        r[rh][c] = rh < nrhs ? __ldcg(b + (long long)rh * Np + i * TB + c) : 0.0;
    }
    __syncthreads();
    // ---- backward ----
    const int c = tid & 127, h = tid >> 7;
    for (int k = a.nb - 1; k >= 0; k--) {
        if (i == k) {
            const double* Li = a.Linv + (long long)k * TB * TB;
            double s0 = 0.0, s1 = 0.0;
            for (int m = c + h; m < TB; m += 2) {
                double l = Li[m * TB + c];
                s0 = fma(l, r[0][m], s0);
                s1 = fma(l, r[1][m], s1);
            }
            part[0][h][c] = s0;
            part[1][h][c] = s1;
            __syncthreads();
            if (h == 0) {
                b[k * TB + c] = part[0][0][c] + part[0][1][c];
                if (nrhs > 1) b[Np + k * TB + c] = part[1][0][c] + part[1][1][c];
            }
        }
        grid.sync();
        if (i < k) {
            for (int q = tid; q < 2 * TB; q += NTHREADS) {
                int rh = q >> 7, cc = q & 127;
                yk[rh][cc] = rh < nrhs ? __ldcg(b + (long long)rh * Np + k * TB + cc) : 0.0;
            }
            __syncthreads();
            const double* T = L + (long long)k * TB * Np + (long long)i * TB;  // L[k, i], used transposed
            double s0 = 0.0, s1 = 0.0;
            for (int m = h; m < TB; m += 2) {
                double l = T[(long long)m * Np + c];
                s0 = fma(l, yk[0][m], s0);
                s1 = fma(l, yk[1][m], s1);
            }
            part[0][h][c] = s0;
            part[1][h][c] = s1;
            __syncthreads();
            if (h == 0) {
                r[0][c] -= part[0][0][c] + part[0][1][c];
                r[1][c] -= part[1][0][c] + part[1][1][c];
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// Dataflow TRSV for ONE large problem: CTA i owns row block i, all nb CTAs co-resident (cooperative launch).  Instead of a
// grid barrier per block step (k_trsv_big: ~15 us per step, 1 ms per solve at nb = 32, profiles/r02_cfg1_launches_v1.csv)
// the blocks are chained by flags: CTA i streams the tiles L[i,k] (forward) / L[k,i] (backward) in order, has the NEXT
// tile's loads in registers before it waits for y_k / x_k, and publishes its own block with a release store.  The inverse
// of its diagonal block sits in shared memory for the whole kernel.  Critical path per block step: flag hop + one 1 KB
// vector read + a 128x128 GEMV from registers + a 128x128 GEMV from shared memory.
// ------------------------------------------------------------------------------------------------------------
constexpr int LDI = TB + 1;  // smem stride of the diagonal inverse (conflict-free for row- and column-wise access)
__device__ __forceinline__ void flag_wait(const int* f) {
    if (threadIdx.x == 0) {
        int v;
        do {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        } while (v == 0);
    }
    __syncthreads();
}
__device__ __forceinline__ void flag_set(int* f) {
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(f), "r"(1) : "memory");
}

__global__ void __launch_bounds__(NTHREADS, 1) k_trsv_flow(const __grid_constant__ CholArgs a, double* b, int nrhs,
                                                          int fwd_done, int* flags /* [2][nb], zero on entry */) {
    extern __shared__ __align__(16) double sm[];
    double* Li = sm;               // [128][LDI] inverse of the diagonal block
    double* rs = Li + TB * LDI;    // [2][128] this block's running right-hand side
    double* vs = rs + 2 * TB;      // [2][128] the published block of the current step
    double* part = vs + 2 * TB;    // [4][2][128] partial sums
    const int tid = threadIdx.x;
    const int i = blockIdx.x, nb = a.nb;
    const long long Np = a.Np;
    const double* L = a.G;
    if (__ldcg(a.info) != 0) return;  // broken factorisation (set before this launch): every CTA leaves
    for (int idx = tid; idx < TB * TB; idx += NTHREADS) {
        const int r = idx >> 7, c = idx & 127;
        Li[r * LDI + c] = a.Linv[(long long)i * TB * TB + idx];
    }
    for (int q = tid; q < 2 * TB; q += NTHREADS) rs[q] = (q >> 7) < nrhs ? b[(long long)(q >> 7) * Np + i * TB + (q & 127)] : 0.0;
    __syncthreads();
    if (!fwd_done) {
        // ---- forward: r_i -= L[i,k] y_k for k < i, then y_i = Linv_ii r_i ----
        const int row = tid >> 1, half = tid & 1;
        const double* Lrow = L + ((long long)i * TB + row) * Np + half * 64;
        for (int k = 0; k < i; k++) {
            double2 tl[32];
#pragma unroll
            for (int j = 0; j < 32; j++) tl[j] = __ldg(reinterpret_cast<const double2*>(Lrow + (long long)k * TB) + j);
            flag_wait(flags + k);
            for (int q = tid; q < 2 * TB; q += NTHREADS)
                vs[q] = (q >> 7) < nrhs ? __ldcg(b + (long long)(q >> 7) * Np + k * TB + (q & 127)) : 0.0;
            __syncthreads();
            double s0, s1;
            {
                double e0[4] = {0.0, 0.0, 0.0, 0.0}, e1[4] = {0.0, 0.0, 0.0, 0.0};  // 4 chains: latency and rounding
#pragma unroll
                for (int j = 0; j < 32; j++) {
                    const int c = half * 64 + 2 * j;
                    e0[j & 3] = fma(tl[j].x, vs[c], fma(tl[j].y, vs[c + 1], e0[j & 3]));
                    e1[j & 3] = fma(tl[j].x, vs[TB + c], fma(tl[j].y, vs[TB + c + 1], e1[j & 3]));
                }
                s0 = (e0[0] + e0[1]) + (e0[2] + e0[3]);
                s1 = (e1[0] + e1[1]) + (e1[2] + e1[3]);
            }
            s0 += __shfl_xor_sync(0xffffffffu, s0, 1);
            s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
            if (half == 0) {
                rs[row] -= s0;
                rs[TB + row] -= s1;
            }
            __syncthreads();
        }
        {
            const int r = tid & 127, h = tid >> 7;  // rhs h
            double e[4] = {0.0, 0.0, 0.0, 0.0};
            for (int c = 0; c <= r; c++) e[c & 3] = fma(Li[r * LDI + c], rs[h * TB + c], e[c & 3]);
            const double s = (e[0] + e[1]) + (e[2] + e[3]);
            __syncthreads();
            rs[h * TB + r] = s;  // y_i: also the backward right-hand side of this block
            if (h < nrhs) b[(long long)h * Np + i * TB + r] = s;
        }
        flag_set(flags + i);
    }
    // ---- backward: r_i -= L[k,i]' x_k for k > i, then x_i = Linv_ii' r_i ----
    {
        const int c2 = tid & 63, rq = tid >> 6;
        for (int k = nb - 1; k > i; k--) {
            double2 tl[32];
            const double* T = L + ((long long)k * TB + rq * 32) * Np + (long long)i * TB + 2 * c2;
#pragma unroll
            for (int j = 0; j < 32; j++) tl[j] = __ldg(reinterpret_cast<const double2*>(T + (long long)j * Np));
            flag_wait(flags + nb + k);
            for (int q = tid; q < 2 * TB; q += NTHREADS)
                vs[q] = (q >> 7) < nrhs ? __ldcg(b + (long long)(q >> 7) * Np + k * TB + (q & 127)) : 0.0;
            __syncthreads();
            double q00[2] = {0.0, 0.0}, q01[2] = {0.0, 0.0}, q10[2] = {0.0, 0.0}, q11[2] = {0.0, 0.0};
#pragma unroll
            for (int j = 0; j < 32; j++) {
                const double x0 = vs[rq * 32 + j], x1 = vs[TB + rq * 32 + j];
                q00[j & 1] = fma(tl[j].x, x0, q00[j & 1]);
                q01[j & 1] = fma(tl[j].y, x0, q01[j & 1]);
                q10[j & 1] = fma(tl[j].x, x1, q10[j & 1]);
                q11[j & 1] = fma(tl[j].y, x1, q11[j & 1]);
            }
            const double p00 = q00[0] + q00[1], p01 = q01[0] + q01[1];  // [rhs][column of the pair]
            const double p10 = q10[0] + q10[1], p11 = q11[0] + q11[1];
            part[(rq * 2 + 0) * TB + 2 * c2] = p00;
            part[(rq * 2 + 0) * TB + 2 * c2 + 1] = p01;
            part[(rq * 2 + 1) * TB + 2 * c2] = p10;
            part[(rq * 2 + 1) * TB + 2 * c2 + 1] = p11;
            __syncthreads();
            {
                const int c = tid & 127, h = tid >> 7;
                rs[h * TB + c] -= (part[(0 * 2 + h) * TB + c] + part[(1 * 2 + h) * TB + c]) +
                                  (part[(2 * 2 + h) * TB + c] + part[(3 * 2 + h) * TB + c]);
            }
            __syncthreads();
        }
        const int c = tid & 127, h = tid >> 7;
        double e[4] = {0.0, 0.0, 0.0, 0.0};
        for (int m = c; m < TB; m++) e[m & 3] = fma(Li[m * LDI + c], rs[h * TB + m], e[m & 3]);
        const double s = (e[0] + e[1]) + (e[2] + e[3]);
        if (h < nrhs) b[(long long)h * Np + i * TB + c] = s;
        flag_set(flags + nb + i);
    }
}
constexpr size_t TRSV_FLOW_SMEM = sizeof(double) * (TB * LDI + 2 * TB + 2 * TB + 8 * TB);

// ------------------------------------------------------------------------------------------------------------
// (L L') X = B for many right-hand sides that share one factor: one CTA per (problem, chunk of CC channels), B[p][c][Np]
// solved in place.  Per 128-block step
//   forward   R_k = B_k - sum_{i<k} L_ki Y_i,    Y_k = Linv_kk R_k
//   backward  R_k = Y_k - sum_{r>k} L_rk' X_r,   X_k = Linv_kk' R_k
// every product is a 128 x CC panel on DMMA m8n8k4 (warp w: rows 16w .. 16w+15, all CC columns).  The k-dimension streams
// through a two-stage cp.async ring of 32-wide chunks: forward chunks of L are [128 rows][32 columns] (fragments as in
// gram.cu), backward chunks [32 rows][128 columns] read transposed (row stride == 4 mod 16 doubles: conflict-free per half
// warp).  The kept inverses Linv_kk are read lower-triangle only (their upper part is not specified).  L is read once
// per problem and chunk: the solve is bound by those 2 (Np^2 / 2 + nb 128^2) 8 bytes.
// ------------------------------------------------------------------------------------------------------------
constexpr int TS_LDF = KC + 4;       // forward chunk row stride (== LDT)
constexpr int TS_LDB = TB + 4;       // backward chunk / R panel row stride
constexpr int TS_LST = TB * TS_LDF;  // doubles per L stage (>= KC * TS_LDB)
template <int CC>
constexpr size_t trsm_multi_smem_d() {
    return 2 * TS_LST + 2 * CC * TS_LDF + CC * TS_LDB;
}

template <int CC>
__global__ void __launch_bounds__(NTHREADS, 2) k_trsm_multi(const __grid_constant__ CholArgs a, double* __restrict__ Bm,
                                                            long long strideB, int C) {
    extern __shared__ __align__(16) double sm[];
    double* sL = sm;                     // [2][TS_LST]
    double* sX = sm + 2 * TS_LST;        // [2][CC][TS_LDF]
    double* sR = sX + 2 * CC * TS_LDF;   // [CC][TS_LDB]: the panel R_k, stored [channel][row]
    constexpr int NT = CC / 8;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int prob = blockIdx.y, c0 = blockIdx.x * CC, nc = min(CC, C - c0);
    const int Np = a.Np, nb = a.nb;
    if (__ldcg(a.info + prob) != 0) return;  // broken factorisation: nothing to solve (the caller re-does the window)
    const double* L = a.G + (long long)prob * a.strideG;
    const double* Li = a.Linv + (long long)prob * a.strideLinv;
    double* X = Bm + (long long)prob * strideB;
    auto xrow = [&](int n) { return X + (long long)(c0 + min(n, nc - 1)) * Np; };  // absent channels re-read the last one
    double acc[2][NT][2];
    const int fr = lane >> 2, fk = lane & 3;

    for (int dir = 0; dir < 2; dir++) {
        const bool fwd = dir == 0;
        for (int s = 0; s < nb; s++) {
            const int k = fwd ? s : nb - 1 - s;
            const int nq = 4 * (fwd ? k : nb - 1 - k), total = nq + 4;
            auto issue = [&](int q, int st) {
                double* dL = sL + st * TS_LST;
                if (q < nq) {
                    const int blk = fwd ? q / 4 : k + 1 + q / 4, kc = (q & 3) * KC;
                    if (fwd) {
                        load_tile_async(dL, L + (long long)k * TB * Np + blk * TB + kc, Np, tid);
                    } else {
#pragma unroll
                        for (int i = 0; i < (KC * TB / 2) / NTHREADS; i++) {
                            const int e = tid + i * NTHREADS, row = e >> 6, seg = e & 63;
                            cp_async16(dL + row * TS_LDB + 2 * seg, L + (long long)(blk * TB + kc + row) * Np + k * TB + 2 * seg);
                        }
                    }
                    double* dX = sX + st * CC * TS_LDF;
                    for (int e = tid; e < CC * (KC / 2); e += NTHREADS) {
                        const int n = e / (KC / 2), seg = e % (KC / 2);
                        cp_async16(dX + n * TS_LDF + 2 * seg, xrow(n) + blk * TB + kc + 2 * seg);
                    }
                } else {
                    const int kc = (q - nq) * KC;
                    const double* Lk = Li + (long long)k * TB * TB;
                    if (fwd) {
                        load_tile_async(dL, Lk + kc, TB, tid);
                    } else {
#pragma unroll
                        for (int i = 0; i < (KC * TB / 2) / NTHREADS; i++) {
                            const int e = tid + i * NTHREADS, row = e >> 6, seg = e & 63;
                            cp_async16(dL + row * TS_LDB + 2 * seg, Lk + (long long)(kc + row) * TB + 2 * seg);
                        }
                    }
                }
                cp_async_commit();
            };
#pragma unroll
            for (int i = 0; i < 2; i++)
#pragma unroll
                for (int j = 0; j < NT; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
            issue(0, 0);
            for (int q = 0; q < total; q++) {
                if (q + 1 < total)
                    issue(q + 1, (q + 1) & 1);
                else
                    cp_async_commit();
                cp_async_wait<1>();
                __syncthreads();
                const bool diag = q >= nq;
                if (q == nq) {  // R_k = rhs block - accumulated products, into shared memory [channel][row]
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        const int m = 16 * w + 8 * i + fr;
#pragma unroll
                        for (int j = 0; j < NT; j++)
#pragma unroll
                            for (int e = 0; e < 2; e++) {
                                const int n = 8 * j + 2 * fk + e;
                                sR[n * TS_LDB + m] = __ldcg(xrow(n) + k * TB + m) - acc[i][j][e];
                                acc[i][j][e] = 0.0;
                            }
                    }
                    __syncthreads();
                }
                const double* cL = sL + (q & 1) * TS_LST;
                const double* cX = sX + (q & 1) * CC * TS_LDF;
                const int kq = diag ? (q - nq) * KC : 0;  // column offset of this chunk inside the diagonal block
#pragma unroll
                for (int kk = 0; kk < KC / 4; kk++) {
                    double av[2], bv[NT];
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        const int m = 16 * w + 8 * i + fr, kl = 4 * kk + fk;
                        double v = fwd ? cL[m * TS_LDF + kl] : cL[kl * TS_LDB + m];
                        if (diag && (fwd ? kq + kl > m : m > kq + kl)) v = 0.0;  // outside the lower triangle of Linv_kk
                        av[i] = v;
                    }
#pragma unroll
                    for (int j = 0; j < NT; j++)
                        bv[j] = diag ? sR[(8 * j + fr) * TS_LDB + kq + 4 * kk + fk] : cX[(8 * j + fr) * TS_LDF + 4 * kk + fk];
#pragma unroll
                    for (int i = 0; i < 2; i++)
#pragma unroll
                        for (int j = 0; j < NT; j++) dmma884(acc[i][j][0], acc[i][j][1], av[i], bv[j]);
                }
                __syncthreads();  // this stage is refilled two chunks on
            }
            // Y_k / X_k back into B (read again by the later steps of this CTA)
#pragma unroll
            for (int i = 0; i < 2; i++) {
                const int m = 16 * w + 8 * i + fr;
#pragma unroll
                for (int j = 0; j < NT; j++)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int n = 8 * j + 2 * fk + e;
                        if (n < nc) X[(long long)(c0 + n) * Np + k * TB + m] = acc[i][j][e];
                    }
            }
            __threadfence_block();
            __syncthreads();
        }
    }
}

bool attrs_done[64] = {};  // per device
void set_attrs() {
    int dev = 0;
    cudaGetDevice(&dev);
    if (attrs_done[dev & 63]) return;
    cudaFuncSetAttribute(k_potf2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(POTF2_SMEM_D * sizeof(double)));
    cudaFuncSetAttribute(k_gemm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(4 * TILE_D * sizeof(double)));
    attrs_done[dev & 63] = true;
}

}  // namespace

size_t potf2_smem_bytes() { return POTF2_SMEM_D * sizeof(double); }
size_t gemm_smem_bytes() { return 4 * TILE_D * sizeof(double); }

void launch_diag_prepare(double* G, long long strideG, int Np, int ncc, int zero_first, const double* ridge_dev,
                         double ridge, int nproblems, cudaStream_t st) {
    for (int p0 = 0; p0 < nproblems; p0 += 32768) {
        int np = nproblems - p0 < 32768 ? nproblems - p0 : 32768;
        dim3 grid((Np + 255) / 256, np);
        k_diag_prepare<<<grid, 256, 0, st>>>(G + (long long)p0 * strideG, strideG, Np, ncc, zero_first,
                                             ridge_dev ? ridge_dev + p0 : nullptr, ridge);
    }
}

void launch_max_diag(const double* G, long long strideG, int Np, int ncc, int zero_first, double* out,
                     int nproblems, cudaStream_t st) {
    k_max_diag<<<nproblems, 256, 0, st>>>(G, strideG, Np, ncc, zero_first, out);
}

void launch_potf2(const CholArgs& a, int k, int nproblems, cudaStream_t st) {
    set_attrs();
    k_potf2<<<nproblems, NTHREADS, potf2_smem_bytes(), st>>>(a, k);
}

static CholArgs offset_args(const CholArgs& a, int p0) {
    CholArgs b = a;
    b.G = a.G + (long long)p0 * a.strideG;
    if (a.Y) b.Y = a.Y + (long long)p0 * a.strideY;
    b.Linv = a.Linv + (long long)p0 * a.strideLinv;
    b.info = a.info + p0;
    return b;
}

void launch_gemm(int mode, const CholArgs& a, int k, int ntiles, int nproblems, cudaStream_t st) {
    set_attrs();
    if (ntiles <= 0) return;
    for (int p0 = 0; p0 < nproblems; p0 += 32768) {
        int np = nproblems - p0 < 32768 ? nproblems - p0 : 32768;
        dim3 grid(ntiles, np);
        k_gemm<<<grid, NTHREADS, gemm_smem_bytes(), st>>>(offset_args(a, p0), mode, k);
    }
}

void launch_init_y(const CholArgs& a, int nproblems, cudaStream_t st) {
    dim3 grid(a.nb, nproblems);
    k_init_y<<<grid, 256, 0, st>>>(a);
}

void launch_symmetrize(double* G, long long strideG, int Np, int nproblems, cudaStream_t st) {
    dim3 grid(Np / 32, Np / 32, nproblems);
    k_symmetrize<<<grid, 256, 0, st>>>(G, strideG, Np);
}

void launch_trsv(const CholArgs& a, double* B, long long strideB, int nrhs, int nproblems, cudaStream_t st,
                 bool fwd_done, int* flow_flags) {
    if (nproblems == 1 && a.nb >= 8) {
        int dev = 0, sms = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (a.nb <= sms && flow_flags) {  // all row blocks co-resident: flag-chained dataflow substitution
            static bool flow_attr[64] = {};
            if (!flow_attr[dev & 63]) {
                cudaFuncSetAttribute(k_trsv_flow, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TRSV_FLOW_SMEM);
                flow_attr[dev & 63] = true;
            }
            cudaMemsetAsync(flow_flags, 0, sizeof(int) * 2 * a.nb, st);
            CholArgs aa = a;
            int fd = fwd_done ? 1 : 0;
            void* args[] = {(void*)&aa, (void*)&B, (void*)&nrhs, (void*)&fd, (void*)&flow_flags};
            if (cudaLaunchCooperativeKernel((void*)k_trsv_flow, dim3(a.nb), dim3(NTHREADS), args, TRSV_FLOW_SMEM, st) ==
                cudaSuccess)
                return;
            cudaGetLastError();
        }
        if (a.nb <= sms) {  // all row blocks co-resident: cooperative multi-CTA substitution
            CholArgs aa = a;
            int fd = fwd_done ? 1 : 0;
            void* args[] = {(void*)&aa, (void*)&B, (void*)&nrhs, (void*)&fd};
            if (cudaLaunchCooperativeKernel((void*)k_trsv_big, dim3(a.nb), dim3(NTHREADS), args, 0, st) == cudaSuccess)
                return;
            cudaGetLastError();
        }
    }
    const size_t xs_bytes = sizeof(double) * 2 * (size_t)a.Np;
    if (fwd_done && xs_bytes <= 200 * 1024) {
        static bool attr_done[64] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        if (!attr_done[dev & 63]) {
            cudaFuncSetAttribute(k_trsv_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            attr_done[dev & 63] = true;
        }
        k_trsv_bwd<<<nproblems, TRSV_T, xs_bytes, st>>>(a, B, strideB, nrhs);
        return;
    }
    k_trsv<<<nproblems, NTHREADS, 0, st>>>(a, B, strideB, nrhs, fwd_done ? 1 : 0);
}

template <int CC>
static void launch_trsm_multi_cc(const CholArgs& a, double* B, long long strideB, int C, int nproblems, cudaStream_t st) {
    const size_t smem = trsm_multi_smem_d<CC>() * sizeof(double);
    static bool attr_done[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_done[dev & 63]) {
        cudaFuncSetAttribute(k_trsm_multi<CC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_done[dev & 63] = true;
    }
    for (int p0 = 0; p0 < nproblems; p0 += 32768) {
        const int np = nproblems - p0 < 32768 ? nproblems - p0 : 32768;
        dim3 grid((C + CC - 1) / CC, np);
        k_trsm_multi<CC><<<grid, NTHREADS, smem, st>>>(offset_args(a, p0), B + (long long)p0 * strideB, strideB, C);
    }
}

int trsm_multi_chunk(int C) { return C <= 8 ? 8 : (C <= 16 ? 16 : 32); }

void launch_trsm_multi(const CholArgs& a, double* B, long long strideB, int C, int nproblems, cudaStream_t st) {
    const int cc = trsm_multi_chunk(C);
    if (cc == 8)
        launch_trsm_multi_cc<8>(a, B, strideB, C, nproblems, st);
    else if (cc == 16)
        launch_trsm_multi_cc<16>(a, B, strideB, C, nproblems, st);
    else
        launch_trsm_multi_cc<32>(a, B, strideB, C, nproblems, st);
}

// TRSM of block column k (m tiles), optionally with one step of iterative refinement (CholArgs::trsm_scratch)
static int trsm_column(const CholArgs& a, int k, int m, int nproblems, cudaStream_t st) {
    if (!a.trsm_scratch || nproblems != 1) {
        launch_gemm(GM_TRSM, a, k, m, nproblems, st);
        return 1;
    }
    // keep the pre-TRSM tiles: a 128-wide column panel of G, rows (k+1)*128 .., into the dense scratch
    cudaMemcpy2DAsync(a.trsm_scratch, TB * sizeof(double), a.G + (long long)(k + 1) * TB * a.Np + (long long)k * TB,
                      (size_t)a.Np * sizeof(double), TB * sizeof(double), (size_t)m * TB, cudaMemcpyDeviceToDevice, st);
    CholArgs b = a;
    b.rhs = nullptr;  // the fused forward substitution would use the unrefined tiles: the caller runs the full solve
    launch_gemm(GM_TRSM, b, k, m, 1, st);
    launch_gemm(GM_TRSM_RES, b, k, m, 1, st);
    launch_gemm(GM_TRSM_FIX, b, k, m, 1, st);
    return 3;
}

int potrf(const CholArgs& a, int nproblems, int sms, cudaStream_t st, const Lookahead* la) {
    int launches = 0;
    const int nb = a.nb;
    const bool left = (long long)nproblems * nb >= 2LL * sms;
    if (!left && la && nb >= 4) {
        // right-looking with look-ahead: main stream = potf2 / TRSM / next-panel update, aux = the rest of the update.
        // (Measured in round 2: running the critical path on a separate highest-priority stream and the rest on a lowest-
        // priority one does not help -- cfg1 19.6 ms against 19.4 ms; profiles/r02_summary.md.)
        launch_potf2(a, 0, nproblems, st);
        launches++;
        for (int k = 0; k + 1 < nb; k++) {
            const int m = nb - k - 1;
            launches += trsm_column(a, k, m, nproblems, st) - 1;
            cudaEventRecord(la->e_trsm, st);
            if (k > 0) cudaStreamWaitEvent(st, la->e_rest, 0);  // block column k+1 carries the updates up to k-1
            launch_gemm(GM_SYRK_COL, a, k, m, nproblems, st);
            launch_potf2(a, k + 1, nproblems, st);
            launches += 3;
            if (m > 1) {
                cudaStreamWaitEvent(la->aux, la->e_trsm, 0);
                launch_gemm(GM_SYRK_REST, a, k, (m - 1) * m / 2, nproblems, la->aux);
                launches++;
            }
            cudaEventRecord(la->e_rest, la->aux);
        }
        cudaStreamWaitEvent(st, la->e_rest, 0);
        return launches;
    }
    for (int k = 0; k < nb; k++) {
        if (left && k > 0) {
            launch_gemm(GM_SYRK_LEFT, a, k, nb - k, nproblems, st);
            launches++;
        }
        launch_potf2(a, k, nproblems, st);
        launches++;
        if (k + 1 < nb) {
            launches += trsm_column(a, k, nb - k - 1, nproblems, st);
            if (!left) {
                int m = nb - k - 1;
                launch_gemm(GM_SYRK_RIGHT, a, k, m * (m + 1) / 2, nproblems, st);
                launches++;
            }
        }
    }
    return launches;
}

int trtri(const CholArgs& a, int nproblems, cudaStream_t st) {
    int launches = 0;
    launch_init_y(a, nproblems, st);
    launches++;
    for (int i = 1; i < a.nb; i++) {
        launch_gemm(GM_TRTRI_A, a, i, i, nproblems, st);
        launch_gemm(GM_TRTRI_B, a, i, i, nproblems, st);
        launches += 2;
    }
    return launches;
}

int potri(const CholArgs& a, int nproblems, cudaStream_t st) {
    int launches = trtri(a, nproblems, st);
    launch_gemm(GM_LAUUM, a, 0, a.nb * (a.nb + 1) / 2, nproblems, st);
    launch_symmetrize(a.G, a.strideG, a.Np, nproblems, st);
    return launches + 2;
}

}  // namespace lpvs
