// Device-resident ADMM (src/lasso.jl:136-171) for ls_sparse_spectral / ls_sparse_spectral_lpv.
//
// Setup (once): Gram G (fused synthesis kernel), M = (G + I/mu)^-1 from the blocked Cholesky factor (potrf+potri).
// Loop (persistent cooperative kernel, no host sync): per iteration
//     x  = M * rhs,          rhs = A'y + (z-u)/mu   (LeastSquares)   or   (z-u)/mu - q   (Quadratic, Q13)
//     z  = prox_{mu g}(x+u),  u += x - z,  ||x-z||_2 checked on device every iteration (Q12)
// The x-update is an HBM-bound GEMV over the full symmetric M (8*Np^2 bytes/iteration); the prox, the dual
// update, the next right-hand side and the residual partial sums are fused into the GEMV epilogue of the CTA that
// owns the rows, so element-wise prox operators need ONE grid barrier per iteration.  Group-L2 and top-r (IndBallL0)
// need the whole x first: they run as a second, tiny phase after a barrier.
#include <cooperative_groups.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "ctx.h"

namespace cg = cooperative_groups;

namespace lpvs {

constexpr int ADMM_THREADS = 512;
constexpr int ADMM_WARPS = ADMM_THREADS / 32;

struct AdmmArgs {
    const double* M;
    const float* M32;  // the inverse rounded to single (LPVS_OPT_ADMM_M32: Float32 callers; half the bytes per iteration)
    int Np;
    const double* q;
    double *x, *z, *u, *v;  // Np each (v = x+u scratch for non-elementwise prox)
    double* r;              // [2][Np] right-hand side, double buffered
    double mu;
    int quad;
    int prox;
    double pparam;
    // group prox: members of group g are gmem[goff[g] .. goff[g+1])
    const int* goff;
    const int* gmem;
    int ngroups;
    double* part;  // [2][grid] residual partial sums
    long long max_iters;
    double tol;
    int check_every;
    int rbuf0;  // which r buffer holds the current rhs at entry
    // Fourier problems: reference position of an internal index (tie order of IndBallL0); ref_half = Nf
    int ref_half, zero_first;
    // outputs
    long long* iters_out;
    double* res_out;
    int* conv_out;
    int* rbuf_out;
    // diagnostics (LPVS_ADMM_TRACE=<file>): clock64 stamps, [TRACE_ITERS][grid][8], of iterations trace_it0..
    long long* trace;
    long long trace_it0;
};
constexpr int TRACE_ITERS = 4;
#define ADMM_TR(slot)                                                                            \
    if (a.trace && tid == 0 && it >= a.trace_it0 && it < a.trace_it0 + TRACE_ITERS)             \
        a.trace[((it - a.trace_it0) * gridDim.x + blockIdx.x) * 8 + (slot)] = clock64();

__device__ __forceinline__ double prox_elem(int kind, double v, double gl, double thr0) {
    if (kind == LPVS_PROX_L1) {  // sign(v) max(|v| - mu*lambda, 0)
        double a = fabs(v) - gl;
        return a > 0.0 ? copysign(a, v) : 0.0;
    }
    // NormL0: keep v iff |v| > sqrt(2 mu lambda)
    return fabs(v) > thr0 ? v : 0.0;
}

// reference position ([cos block; -sin block], src/lsfft.jl:36-47) <-> internal tiled index, Fourier problems
__device__ __forceinline__ int admm_ref_to_internal(int j, int half, int zero_first) {
    if (j < half) return (j >> 6) * 128 + (j & 63);
    const int k = j - half + zero_first;
    return (k >> 6) * 128 + 64 + (k & 63);
}
__device__ __forceinline__ int admm_internal_to_ref(int p, int half, int zero_first) {
    const int q = p >> 7, r = p & 127, part = r >> 6, cc = q * 64 + (r & 63);
    if (cc >= half || (zero_first && part == 1 && cc == 0)) return 0x7fffffff;  // dummy column
    return part == 0 ? cc : half + cc - zero_first;
}

__device__ __forceinline__ double next_rhs(const AdmmArgs& a, int i, double z, double u) {
    double w = (z - u) / a.mu;
    return a.quad ? (w - a.q[i]) : (a.q[i] + w);
}

template <bool STREAM>
__device__ __forceinline__ double2 ldm(const double* p) {
    return STREAM ? __ldcs(reinterpret_cast<const double2*>(p)) : __ldg(reinterpret_cast<const double2*>(p));
}

// ---- shared pieces of one ADMM iteration ---------------------------------------------------------------------

// element-wise prox + dual update + next rhs for entry i; returns (x-z)^2
__device__ __forceinline__ double admm_elem_update(const AdmmArgs& a, double* rn, int i, double xi, double gl,
                                                   double thr0) {
    double ui = a.u[i];
    double zi = prox_elem(a.prox, xi + ui, gl, thr0);
    double di = xi - zi;
    ui += di;
    a.z[i] = zi;
    a.u[i] = ui;
    rn[i] = next_rhs(a, i, zi, ui);
    return di * di;
}

// second phase for the prox operators that need the whole x first (x and v = x+u are in global memory, a grid
// barrier has been passed).  Returns this thread's contribution to ||x-z||^2.
__device__ __forceinline__ double admm_phase_nonelem(const AdmmArgs& a, double* rn, int b, int nblocks, int tid,
                                                     int lane, int w, double gl) {
    const int Np = a.Np;
    double d2 = 0.0;
    if (a.prox == LPVS_PROX_GROUP_L2) {
        // warp per group: z_g = max(0, 1 - mu*lambda/||v_g||) v_g ; ungrouped entries stay z = 0
        for (int g = w * nblocks + b; g <= a.ngroups; g += nblocks * ADMM_WARPS) {  // spread over the CTAs first
            if (g == a.ngroups) {
                // pseudo group: entries not covered by any group (Q16) -> z = 0
                const int lo2 = a.goff[a.ngroups], hi2 = a.goff[a.ngroups + 1];
                for (int m = lo2 + lane; m < hi2; m += 32) {
                    int i = a.gmem[m];
                    double xi = __ldcg(a.x + i), ui = a.u[i];
                    double di = xi;
                    ui += di;
                    a.z[i] = 0.0;
                    a.u[i] = ui;
                    rn[i] = next_rhs(a, i, 0.0, ui);
                    d2 += di * di;
                }
                continue;
            }
            const int lo = a.goff[g], hi = a.goff[g + 1];
            double ss = 0.0;
            for (int m = lo + lane; m < hi; m += 32) {
                double vi = __ldcg(a.v + a.gmem[m]);
                ss += vi * vi;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
            double nrm = sqrt(ss);
            double scale = nrm > 0.0 ? fmax(0.0, 1.0 - gl / nrm) : 0.0;
            for (int m = lo + lane; m < hi; m += 32) {
                int i = a.gmem[m];
                double vi = __ldcg(a.v + i), xi = __ldcg(a.x + i), ui = a.u[i];
                double zi = scale * vi;
                double di = xi - zi;
                ui += di;
                a.z[i] = zi;
                a.u[i] = ui;
                rn[i] = next_rhs(a, i, zi, ui);
                d2 += di * di;
            }
        }
    } else if (b == 0) {  // LPVS_PROX_BALL_L0: keep the r largest |v| (ties -> lower index); block 0 only
        __shared__ unsigned hist[256];
        __shared__ unsigned long long s_prefix;
        __shared__ unsigned s_want;
        __shared__ int s_tie_cut;
        const unsigned rkeep = (unsigned)a.pparam;
        if (tid == 0) {
            s_prefix = 0ull;
            s_want = rkeep;
        }
        __syncthreads();
        // radix select (MSB first) of the rkeep-th largest key = bits(|v|)
        for (int pass = 7; pass >= 0 && rkeep > 0 && rkeep < (unsigned)Np; pass--) {
            for (int k = tid; k < 256; k += ADMM_THREADS) hist[k] = 0;
            __syncthreads();
            const unsigned long long hi_mask = pass == 7 ? 0ull : (~0ull << (8 * (pass + 1)));
            const unsigned long long prefix = s_prefix;
            for (int i = tid; i < Np; i += ADMM_THREADS) {
                unsigned long long key = (unsigned long long)__double_as_longlong(fabs(__ldcg(a.v + i)));
                if ((key & hi_mask) == prefix) atomicAdd(&hist[(key >> (8 * pass)) & 255], 1u);
            }
            __syncthreads();
            if (tid == 0) {
                unsigned want = s_want, accn = 0;
                int d = 255;
                for (; d > 0; d--) {
                    if (accn + hist[d] >= want) break;
                    accn += hist[d];
                }
                s_want = want - accn;
                s_prefix = prefix | ((unsigned long long)d << (8 * pass));
            }
            __syncthreads();
        }
        const unsigned long long kth = s_prefix;  // key of the r-th largest
        const unsigned ties_to_take = s_want;     // entries equal to kth that are kept
        // Ties are broken in the REFERENCE's index order -- sortperm(abs.(x), rev=true) is stable over [cos block; sin block]
        // (ProximalOperators IndBallL0) -- not in the order of the internal tiled layout, which interleaves the two blocks
        // in groups of 64 and would keep a different support for Nf > 64.  Usually every tie is kept (the r-th largest is
        // unique): the serial scan in reference order only runs when it is not.
        __shared__ unsigned s_nties;
        if (tid == 0) s_nties = 0u;
        __syncthreads();
        if (rkeep > 0 && rkeep < (unsigned)Np) {
            unsigned mine = 0;
            for (int i = tid; i < Np; i += ADMM_THREADS)
                mine += ((unsigned long long)__double_as_longlong(fabs(__ldcg(a.v + i))) == kth) ? 1u : 0u;
            if (mine) atomicAdd(&s_nties, mine);
        }
        __syncthreads();
        if (tid == 0) {
            int cut = 0x7fffffff;  // reference index of the last tie kept; default: all of them
            if (rkeep > 0 && rkeep < (unsigned)Np && ties_to_take < s_nties) {
                cut = -1;
                unsigned seen = 0;
                const int nref = 2 * a.ref_half - a.zero_first;
                for (int j = 0; j < nref && seen < ties_to_take; j++) {
                    const int i = admm_ref_to_internal(j, a.ref_half, a.zero_first);
                    unsigned long long key = (unsigned long long)__double_as_longlong(fabs(__ldcg(a.v + i)));
                    if (key == kth) {
                        seen++;
                        cut = j;
                    }
                }
            }
            s_tie_cut = cut;
        }
        __syncthreads();
        const int cut = s_tie_cut;
        for (int i = tid; i < Np; i += ADMM_THREADS) {
            double vi = __ldcg(a.v + i), xi = __ldcg(a.x + i), ui = a.u[i];
            unsigned long long key = (unsigned long long)__double_as_longlong(fabs(vi));
            bool keep;
            if (rkeep == 0) keep = false;
            else if (rkeep >= (unsigned)Np) keep = true;
            else keep = key > kth || (key == kth && (cut == 0x7fffffff ||
                                                     admm_internal_to_ref(i, a.ref_half, a.zero_first) <= cut));
            double zi = keep ? vi : 0.0;
            double di = xi - zi;
            ui += di;
            a.z[i] = zi;
            a.u[i] = ui;
            rn[i] = next_rhs(a, i, zi, ui);
            d2 += di * di;
        }
    }
    return d2;
}

// residual partial of this CTA (fixed-order), grid barrier, stop test.  Returns true when ||x-z|| < tol.
__device__ __forceinline__ bool admm_end_iter(const AdmmArgs& a, cg::grid_group& grid, double d2, long long it,
                                              int b, int nblocks, int tid, int lane, int w, double* wsum,
                                              double* s_nxz, double& nxz) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
    if (lane == 0) wsum[w] = d2;
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
        for (int k = 0; k < ADMM_WARPS; k++) s += wsum[k];
        a.part[(it & 1) * nblocks + b] = s;
    }
    grid.sync();
    if ((it + 1) % a.check_every == 0 || it + 1 == a.max_iters) {
        if (w == 0) {  // fixed-order parallel sum: identical in every CTA and every run
            double s = 0.0;
            for (int k = lane; k < nblocks; k += 32) s += __ldcg(a.part + (it & 1) * nblocks + k);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) *s_nxz = sqrt(s);
        }
        __syncthreads();
        nxz = *s_nxz;
        return nxz < a.tol;
    }
    return false;
}

// ---- variant 1: GEMV over the full symmetric M (small problems, M resident in L2) ------------------------------
// STREAM: M does not fit in L2 -> evict-first loads; otherwise let L2 keep it across iterations
template <bool STREAM>
__global__ void __launch_bounds__(ADMM_THREADS, 1) k_admm(const __grid_constant__ AdmmArgs a) {
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) double sm[];
    double* rs = sm;          // Np
    double* red = sm + a.Np;  // [rows_max][ADMM_WARPS]
    __shared__ double wsum[ADMM_WARPS];
    __shared__ double s_nxz;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int nblocks = gridDim.x, b = blockIdx.x;
    const int Np = a.Np;
    // contiguous row ownership
    const int base = Np / nblocks, extra = Np % nblocks;
    const int r0 = b * base + min(b, extra);
    const int nrows = base + (b < extra ? 1 : 0);
    // column chunks of 64 handled by this warp: chunk c = w, w+16, ...
    const int nchunks = Np >> 6;  // Np is a multiple of 128
    const bool elementwise = (a.prox == LPVS_PROX_L1 || a.prox == LPVS_PROX_L0);
    const double gl = a.mu * a.pparam;
    const double thr0 = sqrt(2.0 * a.mu * a.pparam);

    int cur = a.rbuf0;
    long long it = 0;
    int converged = 0;
    double nxz = 0.0;
    for (; it < a.max_iters; it++) {
        const double* rc = a.r + (long long)cur * Np;
        double* rn = a.r + (long long)(cur ^ 1) * Np;
        for (int i = tid; i < Np; i += ADMM_THREADS) rs[i] = __ldcg(rc + i);
        __syncthreads();
        // ---- x rows = M[rows,:] * r, two rows per pass, column chunks striped over the warps ----
        for (int rr = 0; rr < nrows; rr += 2) {
            const bool two = rr + 1 < nrows;
            const double* m0 = a.M + (long long)(r0 + rr) * Np + 2 * lane;
            const double* m1 = two ? m0 + Np : m0;
            double s0 = 0.0, s1 = 0.0, t0 = 0.0, t1 = 0.0;
            int c = w;
            for (; c + 3 * ADMM_WARPS < nchunks; c += 4 * ADMM_WARPS) {
                double2 a0 = ldm<STREAM>(m0 + 64 * c);
                double2 a1 = ldm<STREAM>(m0 + 64 * (c + ADMM_WARPS));
                double2 a2 = ldm<STREAM>(m0 + 64 * (c + 2 * ADMM_WARPS));
                double2 a3 = ldm<STREAM>(m0 + 64 * (c + 3 * ADMM_WARPS));
                double2 b0 = ldm<STREAM>(m1 + 64 * c);
                double2 b1 = ldm<STREAM>(m1 + 64 * (c + ADMM_WARPS));
                double2 b2 = ldm<STREAM>(m1 + 64 * (c + 2 * ADMM_WARPS));
                double2 b3 = ldm<STREAM>(m1 + 64 * (c + 3 * ADMM_WARPS));
                double2 v0 = *reinterpret_cast<const double2*>(rs + 64 * c + 2 * lane);
                double2 v1 = *reinterpret_cast<const double2*>(rs + 64 * (c + ADMM_WARPS) + 2 * lane);
                double2 v2 = *reinterpret_cast<const double2*>(rs + 64 * (c + 2 * ADMM_WARPS) + 2 * lane);
                double2 v3 = *reinterpret_cast<const double2*>(rs + 64 * (c + 3 * ADMM_WARPS) + 2 * lane);
                s0 = fma(a0.x, v0.x, s0); t0 = fma(a0.y, v0.y, t0);
                s1 = fma(b0.x, v0.x, s1); t1 = fma(b0.y, v0.y, t1);
                s0 = fma(a1.x, v1.x, s0); t0 = fma(a1.y, v1.y, t0);
                s1 = fma(b1.x, v1.x, s1); t1 = fma(b1.y, v1.y, t1);
                s0 = fma(a2.x, v2.x, s0); t0 = fma(a2.y, v2.y, t0);
                s1 = fma(b2.x, v2.x, s1); t1 = fma(b2.y, v2.y, t1);
                s0 = fma(a3.x, v3.x, s0); t0 = fma(a3.y, v3.y, t0);
                s1 = fma(b3.x, v3.x, s1); t1 = fma(b3.y, v3.y, t1);
            }
            for (; c < nchunks; c += ADMM_WARPS) {
                double2 a0 = ldm<STREAM>(m0 + 64 * c);
                double2 b0 = ldm<STREAM>(m1 + 64 * c);
                double2 v0 = *reinterpret_cast<const double2*>(rs + 64 * c + 2 * lane);
                s0 = fma(a0.x, v0.x, s0); t0 = fma(a0.y, v0.y, t0);
                s1 = fma(b0.x, v0.x, s1); t1 = fma(b0.y, v0.y, t1);
            }
            s0 += t0;
            s1 += t1;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            }
            if (lane == 0) {
                red[rr * ADMM_WARPS + w] = s0;
                if (two) red[(rr + 1) * ADMM_WARPS + w] = s1;
            }
        }
        __syncthreads();
        // ---- epilogue for the owned rows ----
        double d2 = 0.0;
        if (tid < nrows) {
            const int i = r0 + tid;
            double xi = 0.0;
#pragma unroll
            for (int k = 0; k < ADMM_WARPS; k++) xi += red[tid * ADMM_WARPS + k];
            a.x[i] = xi;
            if (elementwise)
                d2 = admm_elem_update(a, rn, i, xi, gl, thr0);
            else
                a.v[i] = xi + a.u[i];
        }
        if (!elementwise) {
            grid.sync();
            d2 = admm_phase_nonelem(a, rn, b, nblocks, tid, lane, w, gl);
        }
        const bool stop = admm_end_iter(a, grid, d2, it, b, nblocks, tid, lane, w, wsum, &s_nxz, nxz);
        cur ^= 1;
        if (stop) {
            converged = 1;
            it++;
            break;
        }
    }
    if (b == 0 && tid == 0) {
        *a.iters_out = it;
        *a.res_out = nxz;
        *a.conv_out = converged;
        *a.rbuf_out = cur;
    }
}

// ---- variant 2: SYMV over the lower triangle only (4*Np^2 bytes per iteration) ---------------------------------
// Work unit: a segment = up to SEG consecutive 128x128 blocks (I = i0..i1-1) of one block column J of the lower
// triangle.  Warp w owns rows 8w..8w+7 of every block: 16 independent 16-byte loads per lane per block.
//   row part:    y_I[8w+r]  += sum_c M[I,J][8w+r, c] * r_J[c]          (warp shuffle reduction, single writer)
//   column part: y_J[c]     += sum_r M[I,J][r, c] * r_I[r]  (I != J)   (registers across the segment, then one
//                                                                       cross-warp reduction per segment)
// Each CTA accumulates into a private y in shared memory and publishes it; the cross-CTA sum (fixed order) is
// fused with the prox / dual update / next rhs / residual epilogue after one grid barrier.
__device__ __forceinline__ unsigned long long l2_policy(bool keep) {
    unsigned long long pol;
    if (keep)
        asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    else
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ double2 ld_hint(const double* p, unsigned long long pol) {
    double2 v;
    asm volatile("ld.global.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol));
    return v;
}

__device__ __forceinline__ double2 ld_hint(const float* p, unsigned long long pol) {
    float2 v;
    asm volatile("ld.global.L2::cache_hint.v2.f32 {%0,%1}, [%2], %3;" : "=f"(v.x), "=f"(v.y) : "l"(p), "l"(pol));
    return make_double2((double)v.x, (double)v.y);
}
__device__ __forceinline__ double2 ld_ro(const double* p) { return __ldg(reinterpret_cast<const double2*>(p)); }
__device__ __forceinline__ double2 ld_ro(const float* p) {
    const float2 v = __ldg(reinterpret_cast<const float2*>(p));
    return make_double2((double)v.x, (double)v.y);
}

// One 128x128 block of M, this warp's 8 rows (blk -> row 8w, the lane's columns 2*lane, 2*lane+1, 64+2*lane, 65+2*lane):
// row part M[rows, cols] * r_J reduced over the lanes (returned value is valid in lanes with (lane & 3) == 0, for row
// ((lane>>4)&1)*4 + ((lane>>3)&1)*2 + ((lane>>2)&1) of the 8), column part M[rows, cols]' * r_I accumulated into c0..c3.
// 16 independent 16-byte loads per lane.
template <bool HINT, typename MT = double>
__device__ __forceinline__ double symv_block(const MT* blk, long long Np, unsigned long long pol,
                                             const double (&rs8)[8], double2 rj0, double2 rj1, double& c0, double& c1,
                                             double& c2, double& c3, int lane) {
    double2 m0[8], m1[8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        if (HINT) {
            m0[r] = ld_hint(blk + (long long)r * Np, pol);
            m1[r] = ld_hint(blk + (long long)r * Np + 64, pol);
        } else {
            m0[r] = ld_ro(blk + (long long)r * Np);
            m1[r] = ld_ro(blk + (long long)r * Np + 64);
        }
    }
    double s[8];
#pragma unroll
    for (int r = 0; r < 8; r++) {
        s[r] = fma(m0[r].x, rj0.x, fma(m0[r].y, rj0.y, fma(m1[r].x, rj1.x, m1[r].y * rj1.y)));
        c0 = fma(m0[r].x, rs8[r], c0);
        c1 = fma(m0[r].y, rs8[r], c1);
        c2 = fma(m1[r].x, rs8[r], c2);
        c3 = fma(m1[r].y, rs8[r], c3);
    }
    // reduce the 8 row sums over the 32 lanes: 8->4->2->1 values per lane while halving the lane span
#pragma unroll
    for (int r = 0; r < 4; r++) {
        double keep = (lane & 16) ? s[r + 4] : s[r];
        double send = (lane & 16) ? s[r] : s[r + 4];
        s[r] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int r = 0; r < 2; r++) {
        double keep = (lane & 8) ? s[r + 2] : s[r];
        double send = (lane & 8) ? s[r] : s[r + 2];
        s[r] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    {
        double keep = (lane & 4) ? s[1] : s[0];
        double send = (lane & 4) ? s[0] : s[1];
        s[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
    s[0] += __shfl_xor_sync(0xffffffffu, s[0], 2);
    s[0] += __shfl_xor_sync(0xffffffffu, s[0], 1);
    return s[0];
}

constexpr int SEG = 8;
struct SymvPlan {
    const int* seg_j;   // block column
    const int* seg_i0;  // first block row
    const int* seg_i1;  // one past the last block row
    const int* cta_seg; // [grid+1] segment ranges per CTA
    const int* cta_persist;  // [grid] number of leading blocks of each CTA kept L2-resident (evict_last)
    // sparse exchange of the CTA-private partial y: a CTA publishes only the 128-blocks its segments touch
    const int* cta_slot;  // [grid+1] slot range of each CTA
    const int* slot_blk;  // [nslots] which 128-block of y the slot holds
    const int* red_ptr;   // [nb+1] contributors of each 128-block ...
    const int* red_slot;  // ... as slot indices, ordered by CTA (fixed summation order)
    // phase-2 work items of the group prox (ADMM order: groups are contiguous row ranges)
    const int* cta_item;   // [grid+1]
    const int* item_lo;    // first row
    const int* item_hi;    // one past the last row
    const int* item_kind;  // 0 = group (block soft threshold), 1 = rows outside every group (z = 0, Q16)
    double* ypart;         // [nslots][128]
};

// x_i = sum of the published partials of row i; the four q-lanes of a row split the contributor list
__device__ __forceinline__ double symv_row_sum(const SymvPlan& sp, int i, int q) {
    const int R = i >> 7, c = i & 127;
    const int k1 = __ldg(sp.red_ptr + R + 1);
    double t = 0.0;
    for (int k = __ldg(sp.red_ptr + R) + q; k < k1; k += 4)
        t += __ldcg(sp.ypart + (long long)__ldg(sp.red_slot + k) * 128 + c);
    return t;
}

template <typename MT>
__global__ void __launch_bounds__(ADMM_THREADS, 1) k_admm_symv(const __grid_constant__ AdmmArgs a,
                                                               const __grid_constant__ SymvPlan sp) {
    const MT* Mst = sizeof(MT) == 4 ? reinterpret_cast<const MT*>(a.M32) : reinterpret_cast<const MT*>(a.M);
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) double sm[];
    double* ys = sm;             // Np: CTA-private partial y
    double* cred = sm + a.Np;    // [ADMM_WARPS][128] column partials of the current segment
    double* xs = cred + ADMM_WARPS * 128;  // [Np] x of the current group item (group prox only)
    __shared__ double gsum[ADMM_WARPS];
    __shared__ double wsum[ADMM_WARPS];
    __shared__ double s_nxz;
    __shared__ double red4[4][128];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int nblocks = gridDim.x, b = blockIdx.x;
    const int Np = a.Np;
    const bool elementwise = (a.prox == LPVS_PROX_L1 || a.prox == LPVS_PROX_L0);
    const double gl = a.mu * a.pparam;
    const double thr0 = sqrt(2.0 * a.mu * a.pparam);
    // phase-2 row ownership: even split
    const int base = Np / nblocks, extra = Np % nblocks;
    const int r0 = b * base + min(b, extra);
    const int nrows = base + (b < extra ? 1 : 0);
    const int sg0 = sp.cta_seg[b], sg1 = sp.cta_seg[b + 1];
    const int slot0 = sp.cta_slot[b], slot1 = sp.cta_slot[b + 1];
    const int item0 = sp.cta_item[b], item1 = sp.cta_item[b + 1];
    // M is re-read every iteration: a fixed prefix of this CTA's blocks is loaded evict_last so that ~88 MB of M
    // stays in the 126 MB L2 across iterations; the rest streams evict_first
    const int my_persist = sp.cta_persist[b];
    const unsigned long long pol_keep = l2_policy(true), pol_stream = l2_policy(false);

    int cur = a.rbuf0;
    long long it = 0;
    int converged = 0;
    double nxz = 0.0;
    for (; it < a.max_iters; it++) {
        const double* rc = a.r + (long long)cur * Np;
        double* rn = a.r + (long long)(cur ^ 1) * Np;
        ADMM_TR(0)
        for (int sl = slot0 + w; sl < slot1; sl += ADMM_WARPS) {
            const int blk = __ldg(sp.slot_blk + sl);
#pragma unroll
            for (int k = 0; k < 4; k++) ys[blk * 128 + lane + 32 * k] = 0.0;
        }
        __syncthreads();
        // ---- phase 1: this CTA's segments ----
        int bcount = 0;
        for (int sgi = sg0; sgi < sg1; sgi++) {
            const int J = sp.seg_j[sgi], i0 = sp.seg_i0[sgi], i1 = sp.seg_i1[sgi];
            // r_J for the lane's four columns: 2*lane, 2*lane+1, 64+2*lane, 64+2*lane+1
            const double2 rj0 = __ldcg(reinterpret_cast<const double2*>(rc + J * 128 + 2 * lane));
            const double2 rj1 = __ldcg(reinterpret_cast<const double2*>(rc + J * 128 + 64 + 2 * lane));
            double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
            for (int I = i0; I < i1; I++) {
                const MT* blk = Mst + ((long long)I * 128 + 8 * w) * Np + (long long)J * 128 + 2 * lane;
                const unsigned long long pol = (bcount++ < my_persist) ? pol_keep : pol_stream;
                const bool offdiag = I != J;
                double rs8[8];
#pragma unroll
                for (int r = 0; r < 8; r++) rs8[r] = offdiag ? __ldcg(rc + I * 128 + 8 * w + r) : 0.0;
                const double srow = symv_block<true, MT>(blk, Np, pol, rs8, rj0, rj1, c0, c1, c2, c3, lane);
                // lanes with (lane & 3) == 0 hold row index ((lane>>4)&1)*4 + ((lane>>3)&1)*2 + ((lane>>2)&1)
                if ((lane & 3) == 0) {
                    int r = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
                    ys[I * 128 + 8 * w + r] += srow;  // single writer: warp w owns these rows in every block
                }
            }
            // column part of the segment: cross-warp reduction, then into ys[J block]
            cred[w * 128 + 2 * lane] = c0;
            cred[w * 128 + 2 * lane + 1] = c1;
            cred[w * 128 + 64 + 2 * lane] = c2;
            cred[w * 128 + 64 + 2 * lane + 1] = c3;
            __syncthreads();
            if (tid < 128) {
                double t = 0.0;
#pragma unroll
                for (int k = 0; k < ADMM_WARPS; k++) t += cred[k * 128 + tid];
                ys[J * 128 + tid] += t;
            }
            __syncthreads();
        }
        ADMM_TR(1)
        for (int sl = slot0 + w; sl < slot1; sl += ADMM_WARPS) {
            const int blk = __ldg(sp.slot_blk + sl);
            double* yp = sp.ypart + (long long)sl * 128;
#pragma unroll
            for (int k = 0; k < 4; k++) yp[lane + 32 * k] = ys[blk * 128 + lane + 32 * k];
        }
        ADMM_TR(2)
        grid.sync();
        ADMM_TR(3)
        // ---- phase 2: x_i = sum of the published partials (fixed order), then the fused epilogue ----
        double d2 = 0.0;
        if (a.prox != LPVS_PROX_GROUP_L2) {  // evenly split rows
            for (int rb = 0; rb < nrows; rb += 128) {
                const int rl = rb + (tid & 127), q = tid >> 7;
                red4[q][tid & 127] = rl < nrows ? symv_row_sum(sp, r0 + rl, q) : 0.0;
                __syncthreads();
                if (tid < 128 && rl < nrows) {
                    const int i = r0 + rl;
                    const double xi = (red4[0][tid] + red4[1][tid]) + (red4[2][tid] + red4[3][tid]);
                    a.x[i] = xi;
                    if (elementwise)
                        d2 += admm_elem_update(a, rn, i, xi, gl, thr0);
                    else
                        a.v[i] = xi + a.u[i];
                }
                __syncthreads();
            }
        } else {
            // whole groups per CTA: x, v = x+u, ||v_g||, block soft threshold, dual update -- no second barrier.
            // ys was published before the barrier and is free: it holds v of the current item.
            for (int itx = item0; itx < item1; itx++) {
                const int lo = __ldg(sp.item_lo + itx), hi = __ldg(sp.item_hi + itx), kind = __ldg(sp.item_kind + itx);
                for (int rb = lo; rb < hi; rb += 128) {
                    const int i = rb + (tid & 127), q = tid >> 7;
                    red4[q][tid & 127] = i < hi ? symv_row_sum(sp, i, q) : 0.0;
                    __syncthreads();
                    if (tid < 128 && i < hi) {
                        const double xi = (red4[0][tid] + red4[1][tid]) + (red4[2][tid] + red4[3][tid]);
                        a.x[i] = xi;
                        xs[i - lo] = xi;
                        ys[i - lo] = xi + a.u[i];
                    }
                    __syncthreads();
                }
                double scale = 0.0;
                if (kind == 0) {
                    double ss = 0.0;
                    for (int m = tid; m < hi - lo; m += ADMM_THREADS) ss = fma(ys[m], ys[m], ss);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
                    if (lane == 0) gsum[w] = ss;
                    __syncthreads();
                    double tot = 0.0;
#pragma unroll
                    for (int k = 0; k < ADMM_WARPS; k++) tot += gsum[k];
                    const double nrm = sqrt(tot);
                    scale = nrm > 0.0 ? fmax(0.0, 1.0 - gl / nrm) : 0.0;
                }
                for (int m = tid; m < hi - lo; m += ADMM_THREADS) {
                    const int i = lo + m;
                    const double xi = xs[m], zi = scale * ys[m];
                    double ui = a.u[i];
                    const double di = xi - zi;
                    ui += di;
                    a.z[i] = zi;
                    a.u[i] = ui;
                    rn[i] = next_rhs(a, i, zi, ui);
                    d2 += di * di;
                }
                __syncthreads();
            }
        }
        ADMM_TR(4)
        if (a.prox == LPVS_PROX_BALL_L0) grid.sync();
        ADMM_TR(5)
        if (a.prox == LPVS_PROX_BALL_L0) d2 = admm_phase_nonelem(a, rn, b, nblocks, tid, lane, w, gl);
        ADMM_TR(6)
        const bool stop = admm_end_iter(a, grid, d2, it, b, nblocks, tid, lane, w, wsum, &s_nxz, nxz);
        ADMM_TR(7)
        cur ^= 1;
        if (stop) {
            converged = 1;
            it++;
            break;
        }
    }
    if (b == 0 && tid == 0) {
        *a.iters_out = it;
        *a.res_out = nxz;
        *a.conv_out = converged;
        *a.rbuf_out = cur;
    }
}

// ---- variant 3: one CTA per window, many windows per launch (ls_windowpsd/csd/cohere with estimator =
// ls_sparse_spectral, src/lsfft.jl:121 -> src/lasso.jl:105-126).  The windows are independent ADMM problems with
// their own stop test; both channels of a window share M = (A'WA + I/mu)^-1, so one pass over M serves two
// right-hand sides.  No grid barrier: everything a window needs lives in its CTA.
struct AdmmBatchArgs {
    const double* M;      // [nw] Np x Np full symmetric
    long long strideM;
    double* vecs;         // [nw][nrhs][7 Np]: q, x, z, u, v, r0, r1
    int Np, nrhs;
    double mu;
    int quad, prox;
    double pparam;
    int ref_half, zero_first;  // tie order of IndBallL0 (see AdmmArgs)
    long long max_iters;
    double tol;
    long long* iters_out;  // [nw][nrhs]
    double* res_out;       // [nw][nrhs]
};

__global__ void __launch_bounds__(ADMM_THREADS, 1) k_admm_batch(const __grid_constant__ AdmmBatchArgs ba) {
    extern __shared__ __align__(16) double sm[];
    const int Np = ba.Np, nrhs = ba.nrhs;
    double* rs = sm;            // [2][Np] current right-hand sides
    double* xs = sm + 2 * Np;   // [2][Np] x of this iteration
    __shared__ double wsum[2][ADMM_WARPS];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int wdx = blockIdx.x;
    const double* M = ba.M + (long long)wdx * ba.strideM;
    AdmmArgs ch[2];
#pragma unroll
    for (int c = 0; c < 2; c++) {
        double* v = ba.vecs + ((long long)wdx * nrhs + (c < nrhs ? c : 0)) * 7 * Np;
        ch[c] = AdmmArgs{};
        ch[c].Np = Np;
        ch[c].q = v;
        ch[c].x = v + Np;
        ch[c].z = v + 2 * Np;
        ch[c].u = v + 3 * Np;
        ch[c].v = v + 4 * Np;
        ch[c].r = v + 5 * Np;
        ch[c].mu = ba.mu;
        ch[c].quad = ba.quad;
        ch[c].prox = ba.prox;
        ch[c].pparam = ba.pparam;
        ch[c].ref_half = ba.ref_half;
        ch[c].zero_first = ba.zero_first;
    }
    const bool elementwise = (ba.prox == LPVS_PROX_L1 || ba.prox == LPVS_PROX_L0);
    const double gl = ba.mu * ba.pparam;
    const double thr0 = sqrt(2.0 * ba.mu * ba.pparam);
    bool active[2] = {true, nrhs > 1};
    long long its[2] = {0, 0};
    double nxz[2] = {0.0, 0.0};
    int cur = 0;
    for (long long it = 0; it < ba.max_iters && (active[0] || active[1]); it++) {
        for (int i = tid; i < Np; i += ADMM_THREADS) {
            rs[i] = __ldcg(ch[0].r + (long long)cur * Np + i);
            rs[Np + i] = active[1] ? __ldcg(ch[1].r + (long long)cur * Np + i) : 0.0;
        }
        __syncthreads();
        // x = M r for both channels: two rows per pass, lanes across the columns
        for (int rr = 2 * w; rr < Np; rr += 2 * ADMM_WARPS) {
            const double* m0 = M + (long long)rr * Np + 2 * lane;
            const double* m1 = m0 + Np;
            double s00 = 0.0, s01 = 0.0, s10 = 0.0, s11 = 0.0;
            for (int c = 0; c < Np; c += 256) {
                double2 a[4], b[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const bool in = c + 64 * k < Np;
                    a[k] = in ? __ldg(reinterpret_cast<const double2*>(m0 + c + 64 * k)) : make_double2(0.0, 0.0);
                    b[k] = in ? __ldg(reinterpret_cast<const double2*>(m1 + c + 64 * k)) : make_double2(0.0, 0.0);
                }
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    if (c + 64 * k < Np) {
                        const double2 v0 = *reinterpret_cast<const double2*>(rs + c + 64 * k + 2 * lane);
                        const double2 v1 = *reinterpret_cast<const double2*>(rs + Np + c + 64 * k + 2 * lane);
                        s00 = fma(a[k].x, v0.x, s00); s00 = fma(a[k].y, v0.y, s00);
                        s10 = fma(b[k].x, v0.x, s10); s10 = fma(b[k].y, v0.y, s10);
                        s01 = fma(a[k].x, v1.x, s01); s01 = fma(a[k].y, v1.y, s01);
                        s11 = fma(b[k].x, v1.x, s11); s11 = fma(b[k].y, v1.y, s11);
                    }
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                s00 += __shfl_xor_sync(0xffffffffu, s00, o);
                s10 += __shfl_xor_sync(0xffffffffu, s10, o);
                s01 += __shfl_xor_sync(0xffffffffu, s01, o);
                s11 += __shfl_xor_sync(0xffffffffu, s11, o);
            }
            if (lane == 0) {
                xs[rr] = s00;
                xs[rr + 1] = s10;
                xs[Np + rr] = s01;
                xs[Np + rr + 1] = s11;
            }
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < 2; c++) {
            if (!active[c]) continue;  // block-uniform
            double* rn = ch[c].r + (long long)(cur ^ 1) * Np;
            double d2 = 0.0;
            for (int i = tid; i < Np; i += ADMM_THREADS) {
                const double xi = xs[c * Np + i];
                ch[c].x[i] = xi;
                if (elementwise)
                    d2 += admm_elem_update(ch[c], rn, i, xi, gl, thr0);
                else
                    ch[c].v[i] = xi + ch[c].u[i];
            }
            if (!elementwise) {
                __syncthreads();
                d2 = admm_phase_nonelem(ch[c], rn, 0, 1, tid, lane, w, gl);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
            if (lane == 0) wsum[c][w] = d2;
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < 2; c++) {
            if (!active[c]) continue;
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < ADMM_WARPS; k++) s += wsum[c][k];
            nxz[c] = sqrt(s);
            its[c] = it + 1;
            if (nxz[c] < ba.tol) active[c] = false;
        }
        cur ^= 1;
    }
    if (tid == 0) {
        for (int c = 0; c < nrhs; c++) {
            ba.iters_out[(long long)wdx * nrhs + c] = its[c];
            ba.res_out[(long long)wdx * nrhs + c] = nxz[c];
        }
    }
}

// Single-channel variant (PSD, the reference's own windowed-sparse use, test/test_lasso.jl:36): SYMV over the lower
// triangle of the window's inverse -- half the bytes of the GEMV above.  Warp w owns rows 8w..8w+7 of every 128x128
// block; a block column is one segment (column partials stay in registers down the column, one cross-warp reduction per
// column); everything else as k_admm_batch.
__global__ void __launch_bounds__(ADMM_THREADS, 1) k_admm_batch_symv(const __grid_constant__ AdmmBatchArgs ba) {
    extern __shared__ __align__(16) double sm[];
    const int Np = ba.Np, nb = Np >> 7;
    double* rs = sm;                    // [Np] current right-hand side
    double* ys = sm + Np;               // [Np] y = M r
    double* cred = sm + 2 * Np;         // [ADMM_WARPS][128]
    __shared__ double wsum[ADMM_WARPS];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int wdx = blockIdx.x;
    const double* M = ba.M + (long long)wdx * ba.strideM;
    double* v = ba.vecs + (long long)wdx * 7 * Np;
    AdmmArgs ch{};
    ch.Np = Np;
    ch.q = v;
    ch.x = v + Np;
    ch.z = v + 2 * Np;
    ch.u = v + 3 * Np;
    ch.v = v + 4 * Np;
    ch.r = v + 5 * Np;
    ch.mu = ba.mu;
    ch.quad = ba.quad;
    ch.prox = ba.prox;
    ch.pparam = ba.pparam;
    ch.ref_half = ba.ref_half;
    ch.zero_first = ba.zero_first;
    const bool elementwise = (ba.prox == LPVS_PROX_L1 || ba.prox == LPVS_PROX_L0);
    const double gl = ba.mu * ba.pparam;
    const double thr0 = sqrt(2.0 * ba.mu * ba.pparam);
    long long its = 0;
    double nxz = 0.0;
    int cur = 0;
    for (long long it = 0; it < ba.max_iters; it++) {
        for (int i = tid; i < Np; i += ADMM_THREADS) {
            rs[i] = __ldcg(ch.r + (long long)cur * Np + i);
            ys[i] = 0.0;
        }
        __syncthreads();
        for (int J = 0; J < nb; J++) {
            const double2 rj0 = *reinterpret_cast<const double2*>(rs + J * 128 + 2 * lane);
            const double2 rj1 = *reinterpret_cast<const double2*>(rs + J * 128 + 64 + 2 * lane);
            double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
            for (int I = J; I < nb; I++) {
                const double* blk = M + ((long long)I * 128 + 8 * w) * Np + (long long)J * 128 + 2 * lane;
                double rs8[8];
#pragma unroll
                for (int r = 0; r < 8; r++) rs8[r] = I != J ? rs[I * 128 + 8 * w + r] : 0.0;
                const double srow = symv_block<false>(blk, Np, 0ull, rs8, rj0, rj1, c0, c1, c2, c3, lane);
                if ((lane & 3) == 0) {
                    const int r = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
                    ys[I * 128 + 8 * w + r] += srow;  // single writer: warp w owns these rows in every block
                }
            }
            cred[w * 128 + 2 * lane] = c0;
            cred[w * 128 + 2 * lane + 1] = c1;
            cred[w * 128 + 64 + 2 * lane] = c2;
            cred[w * 128 + 64 + 2 * lane + 1] = c3;
            __syncthreads();
            if (tid < 128) {
                double t = 0.0;
#pragma unroll
                for (int k = 0; k < ADMM_WARPS; k++) t += cred[k * 128 + tid];
                ys[J * 128 + tid] += t;
            }
            __syncthreads();
        }
        double* rn = ch.r + (long long)(cur ^ 1) * Np;
        double d2 = 0.0;
        for (int i = tid; i < Np; i += ADMM_THREADS) {
            const double xi = ys[i];
            ch.x[i] = xi;
            if (elementwise)
                d2 += admm_elem_update(ch, rn, i, xi, gl, thr0);
            else
                ch.v[i] = xi + ch.u[i];
        }
        if (!elementwise) {
            __syncthreads();
            d2 = admm_phase_nonelem(ch, rn, 0, 1, tid, lane, w, gl);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
        if (lane == 0) wsum[w] = d2;
        __syncthreads();
        double sres = 0.0;
#pragma unroll
        for (int k = 0; k < ADMM_WARPS; k++) sres += wsum[k];
        nxz = sqrt(sres);
        its = it + 1;
        cur ^= 1;
        if (nxz < ba.tol) break;
    }
    if (tid == 0) {
        ba.iters_out[wdx] = its;
        ba.res_out[wdx] = nxz;
    }
}

// z = copy(x) = x0 (zeros), u = 0, r = rhs(z, u) for every (window, channel); q comes from B[window][channel][Np], window
// stride ldB (2 Np for the two-channel layout, C Np for the matrix path)
__global__ void k_admm_batch_init(const double* __restrict__ B, long long ldB, int Np, int nrhs, double mu, int quad,
                                  double* vecs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Np) return;
    const long long wc = blockIdx.y;  // window * nrhs + channel
    const long long wdx = wc / nrhs, c = wc - wdx * nrhs;
    const double q = B[wdx * ldB + c * Np + i];
    double* v = vecs + wc * 7 * Np;
    v[i] = q;
    v[Np + i] = 0.0;
    v[2 * Np + i] = 0.0;
    v[3 * Np + i] = 0.0;
    v[4 * Np + i] = 0.0;
    v[5 * Np + i] = quad ? -q : q;
    v[6 * Np + i] = 0.0;
}

// z of every (window, channel) back into the [window][channel][Np] solution layout (window stride ldB)
__global__ void k_admm_batch_collect(const double* __restrict__ vecs, int Np, int nrhs, double* __restrict__ B,
                                     long long ldB) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Np) return;
    const long long wc = blockIdx.y;
    const long long wdx = wc / nrhs, c = wc - wdx * nrhs;
    B[wdx * ldB + c * Np + i] = vecs[wc * 7 * Np + 2 * Np + i];
}

// All windows of a batch: M already holds (G + I/mu)^-1 per window, B the weighted right-hand sides A'W[y u].
// On return B holds z (internal layout) per window and channel.
int admm_batch_run(lpvs_ctx* c, const double* d_M, double* d_B, int Np, int nrhs, int nw, int prox, double pparam,
                   double mu, int quad, long long iters, double tol, long long* d_iters, double* d_res, int ref_half,
                   int zero_first) {
    double* vecs = ws<double>(c, BUF_MISC, (size_t)nw * nrhs * 7 * Np);
    if (!vecs) return fail(c, LPVS_E_NOMEM, "out of device memory (ADMM state of %d windows)", nw);
    const size_t smem = sizeof(double) * 4 * (size_t)Np;
    if (smem > 200 * 1024) return fail(c, LPVS_E_UNSUPPORTED, "windowed sparse estimator: Np=%d too large", Np);
    LPVS_CU(c, cudaFuncSetAttribute(k_admm_batch, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (int w0 = 0; w0 < nw; w0 += 16384) {
        const int nn = std::min(16384, nw - w0);
        k_admm_batch_init<<<dim3((Np + 255) / 256, nn * nrhs), 256, 0, c->st>>>(d_B + (long long)w0 * 2 * Np, 2LL * Np, Np,
                                                                               nrhs, mu, quad,
                                                                               vecs + (long long)w0 * nrhs * 7 * Np);
    }
    AdmmBatchArgs ba{};
    ba.M = d_M;
    ba.strideM = (long long)Np * Np;
    ba.vecs = vecs;
    ba.Np = Np;
    ba.nrhs = nrhs;
    ba.mu = mu;
    ba.quad = quad;
    ba.prox = prox;
    ba.pparam = pparam;
    ba.ref_half = ref_half;
    ba.zero_first = zero_first;
    ba.max_iters = iters;
    ba.tol = tol;
    ba.iters_out = d_iters;
    ba.res_out = d_res;
    const size_t smem_symv = sizeof(double) * (2 * (size_t)Np + (size_t)ADMM_WARPS * 128);
    if (nrhs == 1 && c->admm_symv != 0 && smem_symv <= 200 * 1024) {
        // one channel: SYMV over the lower triangle of the window's inverse (4 Np^2 B per window-iteration)
        LPVS_CU(c, cudaFuncSetAttribute(k_admm_batch_symv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_symv));
        k_admm_batch_symv<<<nw, ADMM_THREADS, smem_symv, c->st>>>(ba);
    } else {
        k_admm_batch<<<nw, ADMM_THREADS, smem, c->st>>>(ba);
    }
    for (int w0 = 0; w0 < nw; w0 += 16384) {
        const int nn = std::min(16384, nw - w0);
        k_admm_batch_collect<<<dim3((Np + 255) / 256, nn * nrhs), 256, 0, c->st>>>(
            vecs + (long long)w0 * nrhs * 7 * Np, Np, nrhs, d_B + (long long)w0 * 2 * Np, 2LL * Np);
    }
    c->launches += 3;
    LPVS_CU(c, cudaGetLastError());
    return LPVS_OK;
}

// ---- variant 5: C channels of one window (lpvs_ls_window_matrix_sparse_sums): one CTA per (window, chunk of CC
// channels).  Every channel of the window shares M = (A'WA + I/mu)^-1, so one pass over the lower-triangle 128x128 blocks
// of M per iteration serves the whole chunk: block M_IJ (I >= J) streams through a two-stage cp.async ring of [128 rows]
// [32 columns] chunks (as k_trsm_multi's forward chunks) and every chunk is used twice on DMMA m8n8k4:
//   P1  X_I[128 x CC]      += M_IJ[:, chunk] R_J[chunk, :]    warp w: rows 8w..8w+7, all CC columns, kept in registers
//                                                                  over J = 0..I and stored at the end of block row I
//   P2  X_J[chunk rows, :] += M_IJ[:, chunk]' R_I             (I > J) the chunk read transposed; warp w < 4 CC/8 owns one
//                                                                  8 x 8 output tile over the full k = 128
// X lives in each channel's x vector (global, read-modify-write by a single warp per element and chunk), R in shared
// memory when CC (Np + 4) doubles fit next to the ring, else in the channel's r vector.  Every output element is one
// fixed sequence of DMMA k-steps over the same blocks in the same order, whatever CC, the chunk position or the other
// channels: a channel's z, iteration count and residual are bitwise independent of them.  Each channel has its own stop
// test; a stopped channel's x, z, u and r are no longer written.  Prox and dual update: admm_elem_update /
// admm_phase_nonelem, as k_admm_batch (512 threads: admm_phase_nonelem strides by ADMM_THREADS).
struct AdmmMultiArgs {
    const double* M;  // [nw] Np x Np full symmetric (only the lower-triangle blocks are read)
    long long strideM;
    double* vecs;  // [nw][C][7 Np]: q, x, z, u, v, r, (unused)
    int Np, C;
    double mu;
    int prox;
    double pparam;
    int ref_half, zero_first;
    long long max_iters;
    double tol;
    long long* iters_out;  // [nw][C]
    double* res_out;       // [nw][C]
};
constexpr int AM_LDF = KC + 4;        // chunk row stride (== 4 mod 16: conflict-free fragments, direct and transposed)
constexpr int AM_LST = TB * AM_LDF;   // doubles per ring stage
constexpr int AM_WARPS = ADMM_WARPS;  // 16 warps x 8 rows = one 128-row block

// one [TB x KC] tile into a [TB][LDT] ring stage with NTH threads (load_tile_async for 512-thread CTAs)
template <int NTH>
__device__ __forceinline__ void load_tile_async_n(double* dst, const double* src, long long ld, int tid) {
#pragma unroll
    for (int i = 0; i < (TB * KC / 2) / NTH; i++) {
        const int q = tid + i * NTH, row = q >> 4, seg = q & 15;
        cp_async16(dst + row * LDT + 2 * seg, src + (long long)row * ld + 2 * seg);
    }
}

template <int CC>
__global__ void __launch_bounds__(ADMM_THREADS, 1) k_admm_multi(const __grid_constant__ AdmmMultiArgs ma, int rs_smem) {
    extern __shared__ __align__(16) double sm[];
    double* sM = sm;                // [2][AM_LST]
    double* sR = sm + 2 * AM_LST;   // rs_smem: [CC][Np + 4]
    __shared__ double wsum[CC][AM_WARPS];
    __shared__ int s_stop[CC];
    constexpr int NT = CC / 8;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int fr = lane >> 2, fk = lane & 3;
    const int wdx = blockIdx.y, c0 = blockIdx.x * CC, nc = min(CC, ma.C - c0);
    const int Np = ma.Np, nb = Np / TB;
    const long long vs = 7LL * Np;
    const double* M = ma.M + (long long)wdx * ma.strideM;
    double* V = ma.vecs + ((long long)wdx * ma.C + c0) * vs;  // channel n of the chunk: V + n vs
    const long long ldr = rs_smem ? Np + 4 : vs;
    double* R = rs_smem ? sR : V + 5 * Np;
    auto rcol = [&](int n) { return R + (long long)min(n, nc - 1) * ldr; };  // absent channels re-read the last one
    auto xcol = [&](int n) { return V + (long long)n * vs + Np; };
    auto chan = [&](int n) {
        double* v = V + (long long)n * vs;
        AdmmArgs a{};
        a.Np = Np;
        a.q = v;
        a.x = v + Np;
        a.z = v + 2 * Np;
        a.u = v + 3 * Np;
        a.v = v + 4 * Np;
        a.mu = ma.mu;
        a.quad = 1;
        a.prox = ma.prox;
        a.pparam = ma.pparam;
        a.ref_half = ma.ref_half;
        a.zero_first = ma.zero_first;
        return a;
    };
    if (rs_smem)
        for (int e = tid; e < nc * Np; e += ADMM_THREADS) {
            const int n = e / Np, i = e - n * Np;
            sR[n * ldr + i] = V[n * vs + 5 * Np + i];
        }
    const bool elementwise = (ma.prox == LPVS_PROX_L1 || ma.prox == LPVS_PROX_L0);
    const double gl = ma.mu * ma.pparam;
    const double thr0 = sqrt(2.0 * ma.mu * ma.pparam);
    unsigned active = nc >= 32 ? 0xffffffffu : ((1u << nc) - 1u);
    long long its = 0;  // thread n < nc: channel n's count and residual
    double nxz = 0.0;
    const int total = 2 * nb * (nb + 1);  // chunks of the lower-triangle blocks, row-block major
    __syncthreads();
    for (long long it = 0; it < ma.max_iters && active; it++) {
        auto issue = [&](int I, int J, int q, int st) {
            load_tile_async_n<ADMM_THREADS>(sM + st * AM_LST, M + (long long)I * TB * Np + J * TB + q * KC, Np, tid);
            cp_async_commit();
        };
        double acc[NT][2];
#pragma unroll
        for (int j = 0; j < NT; j++) acc[j][0] = acc[j][1] = 0.0;
        int I = 0, J = 0, q = 0;
        issue(0, 0, 0, 0);
        for (int s = 0; s < total; s++) {
            int nI = I, nJ = J, nq = q + 1;
            if (nq == 4) {
                nq = 0;
                if (++nJ > nI) {
                    nJ = 0;
                    nI++;
                }
            }
            if (s + 1 < total)
                issue(nI, nJ, nq, (s + 1) & 1);
            else
                cp_async_commit();
            cp_async_wait<1>();
            __syncthreads();
            const double* cM = sM + (s & 1) * AM_LST;
            const int kc = J * TB + q * KC;
#pragma unroll
            for (int kk = 0; kk < KC / 4; kk++) {  // P1
                const double av = cM[(8 * w + fr) * AM_LDF + 4 * kk + fk];
#pragma unroll
                for (int j = 0; j < NT; j++) dmma884(acc[j][0], acc[j][1], av, rcol(8 * j + fr)[kc + 4 * kk + fk]);
            }
            if (J < I && w < 4 * NT) {  // P2: rows kc + 8t .. of X_J, columns 8j .., k over the 128 rows of block I
                const int t = w / NT, j = w - t * NT;
                const double* rb = rcol(8 * j + fr) + I * TB;
                double e0 = 0.0, e1 = 0.0, d0 = 0.0, d1 = 0.0;
#pragma unroll 4
                for (int kk = 0; kk < TB / 4; kk += 2) {
                    dmma884(e0, e1, cM[(4 * kk + fk) * AM_LDF + 8 * t + fr], rb[4 * kk + fk]);
                    dmma884(d0, d1, cM[(4 * kk + 4 + fk) * AM_LDF + 8 * t + fr], rb[4 * kk + 4 + fk]);
                }
                e0 += d0;
                e1 += d1;
                const int row = kc + 8 * t + fr, n = 8 * j + 2 * fk;
                if (n < nc && ((active >> n) & 1u)) xcol(n)[row] += e0;
                if (n + 1 < nc && ((active >> (n + 1)) & 1u)) xcol(n + 1)[row] += e1;
            }
            if (J == I && q == 3) {  // block row I complete: X_I = P1 (P2 of the later block rows adds to it)
#pragma unroll
                for (int j = 0; j < NT; j++)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int n = 8 * j + 2 * fk + e;
                        if (n < nc && ((active >> n) & 1u)) xcol(n)[I * TB + 8 * w + fr] = acc[j][e];
                        acc[j][e] = 0.0;
                    }
            }
            __syncthreads();  // this stage is refilled two chunks on; x of this chunk complete
            I = nI;
            J = nJ;
            q = nq;
        }
        // prox, dual update and the next right-hand side of every active channel
        for (int n = 0; n < nc; n++) {
            if (!((active >> n) & 1u)) continue;  // block-uniform
            const AdmmArgs a = chan(n);
            double* rn = R + (long long)n * ldr;
            double d2 = 0.0;
            for (int i = tid; i < Np; i += ADMM_THREADS) {
                const double xi = a.x[i];
                if (elementwise)
                    d2 += admm_elem_update(a, rn, i, xi, gl, thr0);
                else
                    a.v[i] = xi + a.u[i];
            }
            if (!elementwise) {
                __syncthreads();
                d2 = admm_phase_nonelem(a, rn, 0, 1, tid, lane, w, gl);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
            if (lane == 0) wsum[n][w] = d2;
        }
        __syncthreads();
        if (tid < nc && ((active >> tid) & 1u)) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < AM_WARPS; k++) s += wsum[tid][k];
            nxz = sqrt(s);
            its = it + 1;
            s_stop[tid] = nxz < ma.tol;
        }
        __syncthreads();
        for (int n = 0; n < nc; n++)
            if (((active >> n) & 1u) && s_stop[n]) active &= ~(1u << n);
        __syncthreads();
    }
    if (tid < nc) {
        ma.iters_out[(long long)wdx * ma.C + c0 + tid] = its;
        ma.res_out[(long long)wdx * ma.C + c0 + tid] = nxz;
    }
}

// chunk width of the matrix ADMM: the class of k_trsm_multi, narrowed while the shared right-hand sides do not fit next to
// the ring; rs_smem = 0 when even CC = 8 does not fit (Np > 2176): R then stays in each channel's global r vector
constexpr size_t AM_SMEM_CAP = 216 * 1024;
static size_t admm_multi_smem(int cc, int Np, bool rs) {
    return sizeof(double) * (2 * (size_t)AM_LST + (rs ? (size_t)cc * (Np + 4) : 0));
}
void admm_multi_plan(int C, int Np, int* cc, int* rs_smem) {
    int k = trsm_multi_chunk(C);
    while (k > 8 && admm_multi_smem(k, Np, true) > AM_SMEM_CAP) k /= 2;
    *cc = k;
    *rs_smem = admm_multi_smem(k, Np, true) <= AM_SMEM_CAP;
}

template <int CC>
static int launch_admm_multi(lpvs_ctx* c, const AdmmMultiArgs& ma, int nw, int rs) {
    const size_t smem = admm_multi_smem(CC, ma.Np, rs != 0);
    LPVS_CU(c, cudaFuncSetAttribute(k_admm_multi<CC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_admm_multi<CC><<<dim3((ma.C + CC - 1) / CC, nw), ADMM_THREADS, smem, c->st>>>(ma, rs);
    return LPVS_OK;
}

// All windows of a batch, C channels each: M holds (G + I/mu)^-1 per window, B [nw][C][Np] the weighted right-hand sides
// A'W Y; on return B holds z.  d_iters, d_res: [nw][C].
int admm_multi_run(lpvs_ctx* c, const double* d_M, double* d_B, int Np, int C, int nw, int prox, double pparam,
                   double mu, long long iters, double tol, long long* d_iters, double* d_res, int ref_half,
                   int zero_first) {
    const long long ldB = (long long)C * Np;
    double* vecs = ws<double>(c, BUF_MISC, (size_t)nw * C * 7 * Np);
    if (!vecs) return fail(c, LPVS_E_NOMEM, "out of device memory (ADMM state of %d windows x %d channels)", nw, C);
    const int wchunk = std::max(1, std::min(16384, 65535 / C));  // grid.y = windows x channels
    for (int w0 = 0; w0 < nw; w0 += wchunk) {
        const int nn = std::min(wchunk, nw - w0);
        k_admm_batch_init<<<dim3((Np + 255) / 256, nn * C), 256, 0, c->st>>>(d_B + w0 * ldB, ldB, Np, C, mu, 1,
                                                                            vecs + (long long)w0 * C * 7 * Np);
    }
    AdmmMultiArgs ma{};
    ma.M = d_M;
    ma.strideM = (long long)Np * Np;
    ma.vecs = vecs;
    ma.Np = Np;
    ma.C = C;
    ma.mu = mu;
    ma.prox = prox;
    ma.pparam = pparam;
    ma.ref_half = ref_half;
    ma.zero_first = zero_first;
    ma.max_iters = iters;
    ma.tol = tol;
    ma.iters_out = d_iters;
    ma.res_out = d_res;
    int cc, rs, rc;
    admm_multi_plan(C, Np, &cc, &rs);
    if (cc == 8)
        rc = launch_admm_multi<8>(c, ma, nw, rs);
    else if (cc == 16)
        rc = launch_admm_multi<16>(c, ma, nw, rs);
    else
        rc = launch_admm_multi<32>(c, ma, nw, rs);
    if (rc) return rc;
    for (int w0 = 0; w0 < nw; w0 += wchunk) {
        const int nn = std::min(wchunk, nw - w0);
        k_admm_batch_collect<<<dim3((Np + 255) / 256, nn * C), 256, 0, c->st>>>(vecs + (long long)w0 * C * 7 * Np, Np, C,
                                                                                 d_B + w0 * ldB, ldB);
    }
    c->launches += 3;
    LPVS_CU(c, cudaGetLastError());
    return LPVS_OK;
}

// ---- variant 4: ONE problem sharded over the GPUs of a node (one process per GPU, peer memory over NVLink) --------
// Rank r streams a contiguous share of the lower-triangle blocks of M (phase 1 as k_admm_symv); the partial products
// are reduce-scattered to the rank that owns each 128-row block (P2P stores into its receive slots), the owner applies
// prox / dual update and all-gathers the new right-hand side into every rank's copy (P2P stores again).  Two flag
// exchanges per iteration (release/acquire at system scope); no host involvement, no NCCL inside the loop.
// Element-wise prox operators only (L1, L0).
constexpr int SHARD_MAXP = 8;
struct ShardArgs {
    int rank, world;
    int rb[SHARD_MAXP + 1];        // 128-row block ranges owned by the ranks
    double* base[SHARD_MAXP];      // exchange region of every rank (own = local), layout below
    long long off_recv, off_rhs, off_resid, off_flagA, off_flagB, off_abort;  // in doubles
    int rows_max;                  // max rows owned by a rank
    long long it_base;             // iterations done before this launch (flags are absolute iteration counters)
    long long spin_limit;          // clock64 budget of one flag wait
    // exchange v2 (LPVS_OPT_SHARD_EXCHANGE = 1, default): every CTA arrives on counters at every peer instead of
    // "grid barrier -> CTA 0 raises a flag": one grid barrier per iteration instead of three
    int v2;
    long long off_cnt;             // [2] u64 arrival counters: A (partials delivered), B (new rhs + residual partial delivered)
    long long off_resid2;          // [2][SHARD_MAXP][SHARD_MAXGRID] residual partial of every CTA of every rank
    long long off_recv2;           // v3: [2][world][Np] partial of every row from every rank, by iteration parity
};
constexpr int SHARD_MAXGRID = 256;

__device__ __forceinline__ void st_release_sys(long long* p, long long v) {
    asm volatile("st.global.release.sys.b64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ long long ld_acquire_sys(const long long* p) {
    long long v;
    asm volatile("ld.global.acquire.sys.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// Abort protocol (a peer that never shows up must not hang the GPU): every flag wait is bounded by a clock budget and
// never decides anything by itself -- a timeout is only recorded (abort word [1]).  Thread 0 of CTA 0 folds the
// recorded timeouts and the word peers write on their own failure ([0]) into the decision word [2] right BEFORE each
// grid barrier, and every CTA reads [2] right AFTER it, so all CTAs of a rank leave the loop at the same barrier.
__device__ __forceinline__ void shard_wait(const ShardArgs& sh, long long off_flag, long long target, int tid) {
    if (tid < sh.world) {
        const long long* f = reinterpret_cast<const long long*>(sh.base[sh.rank] + off_flag) + tid;
        long long* ab = reinterpret_cast<long long*>(sh.base[sh.rank] + sh.off_abort);
        const long long t0 = clock64();
        while (ld_acquire_sys(f) < target) {
            if (clock64() - t0 > sh.spin_limit || ld_acquire_sys(ab) != 0) {
                atomicExch(reinterpret_cast<unsigned long long*>(ab + 1), 1ull);
                break;
            }
        }
    }
    __syncthreads();
}
// v2: this CTA's stores to every peer are done -> one arrival on each peer's counter.  The bar.sync orders the CTA's stores
// before the arriving threads' release, which is cumulative over them.
__device__ __forceinline__ void shard_arrive(const ShardArgs& sh, int which, int tid) {
    __syncthreads();
    if (tid < sh.world) {
        unsigned long long* cnt = reinterpret_cast<unsigned long long*>(sh.base[tid] + sh.off_cnt) + which;
        asm volatile("red.release.sys.global.add.u64 [%0], %1;" ::"l"(cnt), "l"(1ull) : "memory");
    }
}
// v2: wait until `target` arrivals reached this rank's counter (bounded like shard_wait; a timeout is only recorded)
__device__ __forceinline__ void shard_wait_count(const ShardArgs& sh, int which, unsigned long long target, int tid) {
    if (tid == 0) {
        const long long* cnt = reinterpret_cast<const long long*>(sh.base[sh.rank] + sh.off_cnt) + which;
        long long* ab = reinterpret_cast<long long*>(sh.base[sh.rank] + sh.off_abort);
        const long long t0 = clock64();
        while ((unsigned long long)ld_acquire_sys(cnt) < target) {
            if (clock64() - t0 > sh.spin_limit || ld_acquire_sys(ab) != 0) {
                atomicExch(reinterpret_cast<unsigned long long*>(ab + 1), 1ull);
                break;
            }
        }
    }
    __syncthreads();
}
__device__ __forceinline__ void shard_fold_abort(const ShardArgs& sh, int b, int tid) {
    if (b == 0 && tid == 0) {
        long long* ab = reinterpret_cast<long long*>(sh.base[sh.rank] + sh.off_abort);
        if (ld_acquire_sys(ab) != 0 || ld_acquire_sys(ab + 1) != 0) atomicExch(reinterpret_cast<unsigned long long*>(ab + 2), 1ull);
        __threadfence();
    }
}
__device__ __forceinline__ bool shard_aborted(const ShardArgs& sh) {
    const long long* ab = reinterpret_cast<const long long*>(sh.base[sh.rank] + sh.off_abort);
    return __ldcg(ab + 2) != 0;
}

__global__ void __launch_bounds__(ADMM_THREADS, 1) k_admm_symv_sharded(const __grid_constant__ AdmmArgs a,
                                                                       const __grid_constant__ SymvPlan sp,
                                                                       const __grid_constant__ ShardArgs sh) {
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) double sm[];
    double* ys = sm;
    double* cred = sm + a.Np;
    double* xs = cred + ADMM_WARPS * 128;  // [max_item] x of the current group item (group prox, exchange v3 only)
    __shared__ double wsum[ADMM_WARPS];
    __shared__ double gsum[ADMM_WARPS];
    __shared__ double red4[4][128];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int nblocks = gridDim.x, b = blockIdx.x;
    const int Np = a.Np, P = sh.world, me = sh.rank;
    const int item0 = sp.cta_item[b], item1 = sp.cta_item[b + 1];
    const double gl = a.mu * a.pparam;
    const double thr0 = sqrt(2.0 * a.mu * a.pparam);
    const int sg0 = sp.cta_seg[b], sg1 = sp.cta_seg[b + 1];
    const int slot0 = sp.cta_slot[b], slot1 = sp.cta_slot[b + 1];
    const int my_persist = sp.cta_persist[b];
    const unsigned long long pol_keep = l2_policy(true), pol_stream = l2_policy(false);
    // phase 2a: all Np rows split evenly over this rank's CTAs; phase 2b: the rows this rank owns, split evenly
    const int baseA = Np / nblocks, extraA = Np % nblocks;
    const int a0 = b * baseA + min(b, extraA), an = baseA + (b < extraA ? 1 : 0);
    const int own0 = sh.rb[me] * 128, ownn = (sh.rb[me + 1] - sh.rb[me]) * 128;
    const int baseB = ownn / nblocks, extraB = ownn % nblocks;
    const int b0 = own0 + b * baseB + min(b, extraB), bn = baseB + (b < extraB ? 1 : 0);
    double* mine = sh.base[me];
    int cur = a.rbuf0;
    long long it = 0;
    int converged = 0, failed = 0;
    double nxz = 0.0;
    for (; it < a.max_iters; it++) {
        const long long tick = sh.it_base + it + 1;
        const double* rc = mine + sh.off_rhs + (long long)cur * Np;
        ADMM_TR(0)
        for (int sl = slot0 + w; sl < slot1; sl += ADMM_WARPS) {
            const int blk = __ldg(sp.slot_blk + sl);
#pragma unroll
            for (int k = 0; k < 4; k++) ys[blk * 128 + lane + 32 * k] = 0.0;
        }
        __syncthreads();
        // ---- phase 1: this CTA's segments of this rank's share of the triangle ----
        int bcount = 0;
        for (int sgi = sg0; sgi < sg1; sgi++) {
            const int J = sp.seg_j[sgi], i0 = sp.seg_i0[sgi], i1 = sp.seg_i1[sgi];
            const double2 rj0 = __ldcg(reinterpret_cast<const double2*>(rc + J * 128 + 2 * lane));
            const double2 rj1 = __ldcg(reinterpret_cast<const double2*>(rc + J * 128 + 64 + 2 * lane));
            double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
            for (int I = i0; I < i1; I++) {
                const double* blk = a.M + ((long long)I * 128 + 8 * w) * Np + (long long)J * 128 + 2 * lane;
                const unsigned long long pol = (bcount++ < my_persist) ? pol_keep : pol_stream;
                const bool offdiag = I != J;
                double rs8[8];
#pragma unroll
                for (int r = 0; r < 8; r++) rs8[r] = offdiag ? __ldcg(rc + I * 128 + 8 * w + r) : 0.0;
                const double srow = symv_block<true>(blk, Np, pol, rs8, rj0, rj1, c0, c1, c2, c3, lane);
                if ((lane & 3) == 0) {
                    int r = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
                    ys[I * 128 + 8 * w + r] += srow;
                }
            }
            cred[w * 128 + 2 * lane] = c0;
            cred[w * 128 + 2 * lane + 1] = c1;
            cred[w * 128 + 64 + 2 * lane] = c2;
            cred[w * 128 + 64 + 2 * lane + 1] = c3;
            __syncthreads();
            if (tid < 128) {
                double t = 0.0;
#pragma unroll
                for (int k = 0; k < ADMM_WARPS; k++) t += cred[k * 128 + tid];
                ys[J * 128 + tid] += t;
            }
            __syncthreads();
        }
        for (int sl = slot0 + w; sl < slot1; sl += ADMM_WARPS) {
            const int blk = __ldg(sp.slot_blk + sl);
            double* yp = sp.ypart + (long long)sl * 128;
#pragma unroll
            for (int k = 0; k < 4; k++) yp[lane + 32 * k] = ys[blk * 128 + lane + 32 * k];
        }
        ADMM_TR(1)
        shard_fold_abort(sh, b, tid);
        grid.sync();
        if (shard_aborted(sh)) {
            failed = 1;
            break;
        }
        ADMM_TR(2)
        if (sh.v2 == 2) {
            // ---- exchange v3: ONE cross-GPU step per iteration.  Every rank sends its partial of EVERY row to every peer
            // (an all-reduce by peer stores, Np doubles per peer), then computes x, prox, u and the next right-hand side for
            // all rows itself (redundantly but bit-identically: fixed summation order), so no all-gather and no residual
            // exchange is needed.  Receive buffers alternate with the iteration parity.
            const int par = (int)(tick & 1);
            for (int rb0 = 0; rb0 < an; rb0 += 128) {
                const int rl = rb0 + (tid & 127), q = tid >> 7;
                red4[q][tid & 127] = rl < an ? symv_row_sum(sp, a0 + rl, q) : 0.0;
                __syncthreads();
                if (tid < 128 && rl < an) {
                    const int i = a0 + rl;
                    const double yi = (red4[0][tid] + red4[1][tid]) + (red4[2][tid] + red4[3][tid]);
                    const long long off = sh.off_recv2 + ((long long)(par * P + me)) * Np + i;
                    for (int sdst = 0; sdst < P; sdst++) sh.base[sdst][off] = yi;  // peer (or local) stores over NVLink
                }
                __syncthreads();
            }
            ADMM_TR(3)
            shard_arrive(sh, 0, tid);
            ADMM_TR(4)
            shard_wait_count(sh, 0, (unsigned long long)tick * (unsigned long long)(P * nblocks), tid);
            ADMM_TR(5)
            const int nxt3 = cur ^ 1;
            double d2 = 0.0;
            const double* rbase = mine + sh.off_recv2 + (long long)par * P * Np;
            double* rn3 = mine + sh.off_rhs + (long long)nxt3 * Np;
            if (a.prox == LPVS_PROX_BALL_L0) {
                // IndBallL0 (keep the r largest |x + u|): every rank holds every row after the all-reduce, so each rank runs
                // the single-GPU selection (radix select in block 0, ties in the reference's index order) on its own copy --
                // redundantly and bit-identically, like the element-wise prox; one more local grid barrier, no extra exchange
                for (int r = tid; r < an; r += ADMM_THREADS) {
                    const int i = a0 + r;
                    double xi = 0.0;
                    for (int sr = 0; sr < P; sr++) xi += __ldcg(rbase + (long long)sr * Np + i);
                    a.x[i] = xi;
                    a.v[i] = xi + a.u[i];
                }
                shard_fold_abort(sh, b, tid);
                grid.sync();
                if (shard_aborted(sh)) {
                    failed = 1;
                    break;
                }
                d2 = admm_phase_nonelem(a, rn3, b, nblocks, tid, lane, w, gl);
            } else if (a.prox != LPVS_PROX_GROUP_L2) {
                for (int r = tid; r < an; r += ADMM_THREADS) {
                    const int i = a0 + r;
                    double xi = 0.0;
                    for (int sr = 0; sr < P; sr++) xi += __ldcg(rbase + (long long)sr * Np + i);
                    a.x[i] = xi;
                    double ui = a.u[i];
                    const double zi = prox_elem(a.prox, xi + ui, gl, thr0);
                    const double di = xi - zi;
                    ui += di;
                    a.z[i] = zi;
                    a.u[i] = ui;
                    rn3[i] = next_rhs(a, i, zi, ui);
                    d2 += di * di;
                }
            } else {
                // group prox (src/lasso.jl:53-55): whole groups per CTA in ADMM order, as in k_admm_symv -- every rank holds
                // every row after the all-reduce, so groups never straddle ranks.  ys is free after barrier 1.
                for (int itx = item0; itx < item1; itx++) {
                    const int lo = __ldg(sp.item_lo + itx), hi = __ldg(sp.item_hi + itx), kind = __ldg(sp.item_kind + itx);
                    for (int m = tid; m < hi - lo; m += ADMM_THREADS) {
                        const int i = lo + m;
                        double xi = 0.0;
                        for (int sr = 0; sr < P; sr++) xi += __ldcg(rbase + (long long)sr * Np + i);
                        a.x[i] = xi;
                        xs[m] = xi;
                        ys[m] = xi + a.u[i];
                    }
                    __syncthreads();
                    double scale = 0.0;
                    if (kind == 0) {
                        double ss = 0.0;
                        for (int m = tid; m < hi - lo; m += ADMM_THREADS) ss = fma(ys[m], ys[m], ss);
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
                        if (lane == 0) gsum[w] = ss;
                        __syncthreads();
                        double tot = 0.0;
#pragma unroll
                        for (int k = 0; k < ADMM_WARPS; k++) tot += gsum[k];
                        const double nrm = sqrt(tot);
                        scale = nrm > 0.0 ? fmax(0.0, 1.0 - gl / nrm) : 0.0;
                    }
                    for (int m = tid; m < hi - lo; m += ADMM_THREADS) {
                        const int i = lo + m;
                        const double xi = xs[m], zi = scale * ys[m];
                        double ui = a.u[i];
                        const double di = xi - zi;
                        ui += di;
                        a.z[i] = zi;
                        a.u[i] = ui;
                        rn3[i] = next_rhs(a, i, zi, ui);
                        d2 += di * di;
                    }
                    __syncthreads();
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
            if (lane == 0) wsum[w] = d2;
            __syncthreads();
            if (tid == 0) {
                double sacc = 0.0;
                for (int k = 0; k < ADMM_WARPS; k++) sacc += wsum[k];
                a.part[(it & 1) * nblocks + b] = sacc;
            }
            ADMM_TR(6)
            shard_fold_abort(sh, b, tid);
            grid.sync();
            if (shard_aborted(sh)) {
                failed = 1;
                break;
            }
            ADMM_TR(7)
            if (w == 0) {
                double sacc = 0.0;
                for (int k = lane; k < nblocks; k += 32) sacc += __ldcg(a.part + (it & 1) * nblocks + k);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
                if (lane == 0) wsum[0] = sacc;
            }
            __syncthreads();
            nxz = sqrt(wsum[0]);
            __syncthreads();
            cur = nxt3;
            if ((it + 1) % a.check_every == 0 || it + 1 == a.max_iters) {
                if (nxz < a.tol) {
                    converged = 1;
                    it++;
                    break;
                }
            }
            continue;
        }
        // ---- phase 2a: this rank's partial of every row -> the owner's receive slot [me] (reduce-scatter) ----
        for (int rb0 = 0; rb0 < an; rb0 += 128) {
            const int rl = rb0 + (tid & 127), q = tid >> 7;
            red4[q][tid & 127] = rl < an ? symv_row_sum(sp, a0 + rl, q) : 0.0;
            __syncthreads();
            if (tid < 128 && rl < an) {
                const int i = a0 + rl;
                const double yi = (red4[0][tid] + red4[1][tid]) + (red4[2][tid] + red4[3][tid]);
                const int blk = i >> 7;
                int owner = 0;
                while (blk >= sh.rb[owner + 1]) owner++;
                double* dst = sh.base[owner] + sh.off_recv + (long long)me * sh.rows_max + (i - sh.rb[owner] * 128);
                *dst = yi;  // peer (or local) store over NVLink
            }
            __syncthreads();
        }
        // no per-thread system fence: the stores above happen-before the grid barrier, and the signalling thread's
        // release.sys store after it is cumulative over everything that happened before it
        ADMM_TR(3)
        if (sh.v2) {
            shard_arrive(sh, 0, tid);
            ADMM_TR(4)
            shard_wait_count(sh, 0, (unsigned long long)tick * (unsigned long long)(P * nblocks), tid);
        } else {
            shard_fold_abort(sh, b, tid);
            grid.sync();
            if (shard_aborted(sh)) {
                failed = 1;
                break;
            }
            if (b == 0 && tid < P)
                st_release_sys(reinterpret_cast<long long*>(sh.base[tid] + sh.off_flagA) + me, tick);
            ADMM_TR(4)
            shard_wait(sh, sh.off_flagA, tick, tid);
        }
        ADMM_TR(5)
        // ---- phase 2b: owned rows: x = sum over ranks (fixed order), prox, dual update, new rhs -> every rank ----
        const int nxt = cur ^ 1;
        double d2 = 0.0;
        for (int r = tid; r < bn; r += ADMM_THREADS) {
            const int i = b0 + r;
            const double* rv = mine + sh.off_recv + (i - own0);
            double xi = 0.0;
            for (int s = 0; s < P; s++) xi += __ldcg(rv + (long long)s * sh.rows_max);
            a.x[i] = xi;
            double ui = a.u[i];
            const double zi = prox_elem(a.prox, xi + ui, gl, thr0);
            const double di = xi - zi;
            ui += di;
            a.z[i] = zi;
            a.u[i] = ui;
            const double rn = next_rhs(a, i, zi, ui);
            for (int s = 0; s < P; s++) sh.base[s][sh.off_rhs + (long long)nxt * Np + i] = rn;
            d2 += di * di;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
        if (lane == 0) wsum[w] = d2;
        __syncthreads();
        if (sh.v2) {
            // this CTA's residual partial into its slot at every rank, then one arrival per peer; after the wait every CTA of
            // every rank sums the same P * nblocks slots in the same order -> the same stop decision everywhere
            if (tid < P) {
                double s = 0.0;
                for (int k = 0; k < ADMM_WARPS; k++) s += wsum[k];
                sh.base[tid][sh.off_resid2 + ((long long)(it & 1) * SHARD_MAXP + me) * SHARD_MAXGRID + b] = s;
            }
            ADMM_TR(6)
            shard_arrive(sh, 1, tid);
            shard_wait_count(sh, 1, (unsigned long long)tick * (unsigned long long)(P * nblocks), tid);
            ADMM_TR(7)
            if (w == 0) {
                double s = 0.0;
                for (int r = 0; r < P; r++) {
                    const double* slot = mine + sh.off_resid2 + ((long long)(it & 1) * SHARD_MAXP + r) * SHARD_MAXGRID;
                    double sr = 0.0;
                    for (int k = lane; k < nblocks; k += 32) sr += __ldcg(slot + k);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) sr += __shfl_xor_sync(0xffffffffu, sr, o);
                    s += sr;
                }
                if (lane == 0) wsum[0] = s;
            }
            __syncthreads();
            nxz = sqrt(wsum[0]);
            __syncthreads();
        } else {
            if (tid == 0) {
                double s = 0.0;
                for (int k = 0; k < ADMM_WARPS; k++) s += wsum[k];
                a.part[(it & 1) * nblocks + b] = s;
            }
            shard_fold_abort(sh, b, tid);
            grid.sync();
            if (shard_aborted(sh)) {
                failed = 1;
                break;
            }
            ADMM_TR(6)
            if (b == 0) {
                if (w == 0) {  // this rank's residual partial, fixed order, to every rank; then the flag
                    double s = 0.0;
                    for (int k = lane; k < nblocks; k += 32) s += __ldcg(a.part + (it & 1) * nblocks + k);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                    if (lane < P) {
                        sh.base[lane][sh.off_resid + (it & 1) * SHARD_MAXP + me] = s;
                        st_release_sys(reinterpret_cast<long long*>(sh.base[lane] + sh.off_flagB) + me, tick);
                    }
                }
            }
            shard_wait(sh, sh.off_flagB, tick, tid);
            ADMM_TR(7)
            {
                double s = 0.0;
                for (int k = 0; k < P; k++) s += __ldcg(mine + sh.off_resid + (it & 1) * SHARD_MAXP + k);
                nxz = sqrt(s);
            }
        }
        cur = nxt;
        if ((it + 1) % a.check_every == 0 || it + 1 == a.max_iters) {
            if (nxz < a.tol) {
                converged = 1;
                it++;
                break;
            }
        }
    }
    if (!failed) {  // a timeout in the very last wait has no later barrier to surface at
        shard_fold_abort(sh, b, tid);
        grid.sync();
        if (shard_aborted(sh)) failed = 1;
    }
    if (failed && b == 0 && tid < P)  // tell the peers to stop spinning
        st_release_sys(reinterpret_cast<long long*>(sh.base[tid] + sh.off_abort), 1);
    if (b == 0 && tid == 0) {
        *a.iters_out = it;
        *a.res_out = nxz;
        *a.conv_out = failed ? -1 : converged;
        *a.rbuf_out = cur;
    }
}

// owner -> everyone: final x, z, u rows (so that every rank can answer lpvs_admm_get) -- peer stores, host-synchronised
__global__ void k_shard_broadcast(double* x, double* z, double* u, int row0, int nrows, int Np, ShardArgs sh,
                                  long long off_xzu) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrows) return;
    const int g = row0 + i;
    for (int s = 0; s < sh.world; s++) {
        double* dst = sh.base[s] + off_xzu;
        dst[g] = x[g];
        dst[Np + g] = z[g];
        dst[2 * Np + g] = u[g];
    }
}

__global__ void k_admm_init(const double* __restrict__ q, const double* __restrict__ x0, int Np, double mu,
                            int quad, double* x, double* z, double* u, double* r) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Np) return;
    double v = x0 ? x0[i] : 0.0;
    x[i] = v;
    z[i] = v;  // z = copy(x), u = 0 (src/lasso.jl:146-147)
    u[i] = 0.0;
    double w = v / mu;
    r[i] = quad ? (w - q[i]) : (q[i] + w);
}

// internal vector -> reference order (Fourier: cos block then -sin block; LPV: column-major [Re|Im] un-permuted)
__global__ void k_gather_vec(const double* __restrict__ xin, int nref, int half, int zero_first,
                             const int* __restrict__ pos, double* __restrict__ out) {
    // reference index j: j < half -> real part of complex column j; else imaginary part of column j-half+zero_first
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nref) return;
    int cc, part;
    if (j < half) {
        cc = j;
        part = 0;
    } else {
        cc = j - half + zero_first;
        part = 1;
    }
    const int idx = (cc >> 6) * 128 + part * 64 + (cc & 63);
    out[j] = xin[pos ? pos[idx] : idx];
}

// z = prox_{gamma g}(v) with the loop's own device routines (parity entry lpvs_prox_fourier), one CTA
__global__ void __launch_bounds__(ADMM_THREADS, 1) k_prox_only(const __grid_constant__ AdmmArgs a, double* rn) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const double gl = a.mu * a.pparam, thr0 = sqrt(2.0 * a.mu * a.pparam);
    if (a.prox == LPVS_PROX_L1 || a.prox == LPVS_PROX_L0) {
        for (int i = tid; i < a.Np; i += ADMM_THREADS) a.z[i] = prox_elem(a.prox, a.v[i], gl, thr0);
    } else {
        admm_phase_nonelem(a, rn, 0, 1, tid, lane, w, gl);
    }
}

__global__ void k_to_float(const double* __restrict__ in, float* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)in[i];
}

// ADMM order: Mp[p][q] = M[order[p]][order[q]] (M symmetric), vp[p] = v[order[p]]
__global__ void k_permute_sym(const double* __restrict__ M, double* __restrict__ Mp, const int* __restrict__ order,
                              int Np) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (q < Np) Mp[(long long)p * Np + q] = M[(long long)order[p] * Np + order[q]];
}
__global__ void k_permute_vec(const double* __restrict__ v, double* __restrict__ vp, const int* __restrict__ order,
                              int Np) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < Np) vp[p] = v[order[p]];
}

}  // namespace lpvs

using namespace lpvs;

struct lpvs_admm {
    lpvs_ctx* ctx = nullptr;
    int kind = 0;  // 0 fourier, 1 lpv
    int Np = 0, ncc = 0, zero_first = 0, nref = 0, half = 0;
    int prox = 0;
    double pparam = 0.0, mu = 0.05;
    int quad = 0;
    // LPV bookkeeping for the result permutation
    int lpv_nf = 0, lpv_nvv = 0;
    double* M = nullptr;
    double* vecs = nullptr;  // q, x, z, u, v, r[2]
    int* goff = nullptr;
    int* gmem = nullptr;
    int ngroups = 0;
    double* part = nullptr;
    long long* d_iters = nullptr;  // [iters][res as double bits][conv][rbuf] packed below
    double* d_res = nullptr;
    int* d_flags = nullptr;
    // SYMV variant (lower triangle only)
    int symv = 0;
    float* M32 = nullptr;    // LPVS_OPT_ADMM_M32: the inverse rounded to single, replaces M in the SYMV loop
    int* seg_buf = nullptr;  // all SymvPlan index tables, one allocation
    int nseg = 0;
    size_t off_cta_seg = 0, off_persist = 0, off_cta_slot = 0, off_slot_blk = 0, off_red_ptr = 0, off_red_slot = 0,
           off_cta_item = 0, off_item_lo = 0, off_item_hi = 0, off_item_kind = 0;
    int max_item = 0;  // longest phase-2 item (rows) of the group prox
    // ADMM order (group prox): position p of the loop vectors holds internal index order[p]; pos is the inverse
    std::vector<int> h_order, h_goff;
    int* d_order = nullptr;
    int* d_pos = nullptr;
    // one problem sharded over several GPUs (k_admm_symv_sharded): exchange region + the peers' mappings of theirs
    int shard_rank = 0, shard_world = 1, shard_connected = 0;
    double* xchg = nullptr;
    double* peer_base[8] = {};
    int shard_rb[9] = {};
    long long off_recv = 0, off_rhs = 0, off_resid = 0, off_flagA = 0, off_flagB = 0, off_abort = 0, off_xzu = 0;
    long long off_cnt = 0, off_resid2 = 0, off_recv2 = 0;
    int shard_rows_max = 0;
    double* ypart = nullptr;
    int rbuf = 0;
    int grid = 0;
    int64_t iters_total = 0;
    double residual = INFINITY;
    int converged = 0;
    double last_ms = 0.0;
    int64_t last_iters = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
};

namespace lpvs {

static void admm_release(lpvs_admm* h) {
    if (!h) return;
    auto& live = h->ctx->live_admm;
    live.erase(std::remove(live.begin(), live.end(), h), live.end());
    cudaSetDevice(h->ctx->device);
    cudaStreamSynchronize(h->ctx->st);
    cudaFree(h->M);
    cudaFree(h->M32);
    cudaFree(h->vecs);
    cudaFree(h->goff);
    cudaFree(h->gmem);
    cudaFree(h->part);
    cudaFree(h->d_iters);
    cudaFree(h->d_res);
    cudaFree(h->d_flags);
    cudaFree(h->seg_buf);
    cudaFree(h->ypart);
    cudaFree(h->d_order);
    cudaFree(h->d_pos);
    for (int sidx = 0; sidx < h->shard_world; sidx++)
        if (sidx != h->shard_rank && h->peer_base[sidx]) cudaIpcCloseMemHandle(h->peer_base[sidx]);
    cudaFree(h->xchg);
    if (h->e0) cudaEventDestroy(h->e0);
    if (h->e1) cudaEventDestroy(h->e1);
    delete h;
}

static size_t admm_smem(int Np, int rows_max) { return sizeof(double) * ((size_t)Np + (size_t)rows_max * ADMM_WARPS); }
static size_t admm_smem_symv(int Np, int max_item) {
    return sizeof(double) * ((size_t)Np + (size_t)ADMM_WARPS * 128 + (size_t)max_item);
}

// Phase-2 work items of the group prox: whole groups (ADMM order), the rows outside every group in 128-row pieces;
// longest first onto the least loaded CTA.  Returns the longest item.
struct GroupItems {
    std::vector<int> cta_item, lo, hi, kind;
    int max_item = 0;
};
static GroupItems build_group_items(const lpvs_admm* h, int grid) {
    GroupItems gi;
    gi.cta_item.assign((size_t)grid + 1, 0);
    if (h->prox != LPVS_PROX_GROUP_L2) return gi;
    std::vector<int> ilo, ihi, ikind;
    const int ng = h->ngroups;
    for (int g = 0; g < ng; g++)
        if (h->h_goff[g + 1] > h->h_goff[g]) {
            ilo.push_back(h->h_goff[g]);
            ihi.push_back(h->h_goff[g + 1]);
            ikind.push_back(0);
        }
    for (int r = h->h_goff[ng]; r < h->h_goff[ng + 1]; r += 128) {
        ilo.push_back(r);
        ihi.push_back(std::min(r + 128, h->h_goff[ng + 1]));
        ikind.push_back(1);
    }
    std::vector<int> idx(ilo.size());
    for (size_t k = 0; k < idx.size(); k++) idx[k] = (int)k;
    std::stable_sort(idx.begin(), idx.end(), [&](int x, int y) { return ihi[x] - ilo[x] > ihi[y] - ilo[y]; });
    std::vector<long long> load((size_t)grid, 0);
    std::vector<std::vector<int>> per((size_t)grid);
    for (int k : idx) {
        int best = 0;
        for (int b2 = 1; b2 < grid; b2++)
            if (load[b2] < load[best]) best = b2;
        per[best].push_back(k);
        load[best] += ihi[k] - ilo[k] + 32;  // + a fixed per-item cost
        gi.max_item = std::max(gi.max_item, ihi[k] - ilo[k]);
    }
    for (int b2 = 0; b2 < grid; b2++) {
        gi.cta_item[b2] = (int)gi.lo.size();
        for (int k : per[b2]) {
            gi.lo.push_back(ilo[k]);
            gi.hi.push_back(ihi[k]);
            gi.kind.push_back(ikind[k]);
        }
    }
    gi.cta_item[grid] = (int)gi.lo.size();
    return gi;
}

// SYMV plan for the blocks [tb, te) of the lower triangle (block-column-major order; the whole triangle on one GPU, a
// contiguous share of it when one problem is sharded over several): segments per CTA, L2-resident counts, the sparse
// partial-y exchange tables and the group items.  Replaces any previous plan of the handle.
static int build_symv_plan(lpvs_ctx* c, lpvs_admm* h, const GroupItems& gitems, long long tb, long long te) {
    const int Np = h->Np, nb = Np / TB;
    const int grid = c->sms;
    const long long Tr = te - tb;
    cudaFree(h->seg_buf);
    cudaFree(h->ypart);
    h->seg_buf = nullptr;
    h->ypart = nullptr;
    {
        // blocks of the lower triangle in block-column-major order, split evenly over the CTAs, then cut into
        // segments (same block column, <= SEG blocks)
        std::vector<int> sj, si0, si1, cta(grid + 1, 0);
        std::vector<int> colstart(nb + 1, 0);
        for (int J = 0; J < nb; J++) colstart[J + 1] = colstart[J] + (nb - J);
        int J = 0;
        for (int cta_i = 0; cta_i < grid; cta_i++) {
            long long t0 = tb + Tr * cta_i / grid, t1 = tb + Tr * (cta_i + 1) / grid;
            cta[cta_i] = (int)sj.size();
            long long t = t0;
            while (t < t1) {
                while (colstart[J + 1] <= t) J++;
                int I = J + (int)(t - colstart[J]);
                long long run = std::min<long long>(std::min<long long>(t1 - t, colstart[J + 1] - t), SEG);
                sj.push_back(J);
                si0.push_back(I);
                si1.push_back(I + (int)run);
                t += run;
            }
        }
        cta[grid] = (int)sj.size();
        h->nseg = (int)sj.size();
        // L2-resident share: 88 MB of blocks spread evenly over the CTAs
        std::vector<int> persist(grid, 0);
        {
            const double keep_bytes = 88.0 * 1024 * 1024, blk_bytes = 128.0 * 128.0 * (h->M32 ? 4.0 : 8.0);
            const double frac = std::min(1.0, keep_bytes / ((double)Tr * blk_bytes));
            for (int cta_i = 0; cta_i < grid; cta_i++) {
                long long nblk = Tr * (cta_i + 1) / grid - Tr * cta_i / grid;
                // rounded, not truncated: a CTA that owns one block more keeps one block more in L2, so the number
                // of blocks STREAMED from HBM -- what phase 1 waits for -- is the same for every CTA
                persist[cta_i] = (int)std::lround(frac * (double)nblk);
            }
        }
        // sparse exchange: slots = the 128-blocks of y each CTA touches (block column J and block rows I of its
        // segments); contributor lists per block, ordered by CTA
        std::vector<int> cta_slot(grid + 1, 0), slot_blk;
        std::vector<std::vector<int>> contrib((size_t)nb);
        {
            std::vector<int> seen((size_t)nb, -1);
            for (int cta_i = 0; cta_i < grid; cta_i++) {
                cta_slot[cta_i] = (int)slot_blk.size();
                auto touch = [&](int blk) {
                    if (seen[blk] == cta_i) return;
                    seen[blk] = cta_i;
                    contrib[blk].push_back((int)slot_blk.size());
                    slot_blk.push_back(blk);
                };
                for (int sgi = cta[cta_i]; sgi < cta[cta_i + 1]; sgi++) {
                    touch(sj[sgi]);
                    for (int I = si0[sgi]; I < si1[sgi]; I++) touch(I);
                }
            }
            cta_slot[grid] = (int)slot_blk.size();
        }
        std::vector<int> red_ptr(nb + 1, 0), red_slot;
        for (int R = 0; R < nb; R++) {
            red_ptr[R] = (int)red_slot.size();
            red_slot.insert(red_slot.end(), contrib[R].begin(), contrib[R].end());
        }
        red_ptr[nb] = (int)red_slot.size();
        std::vector<int> all;
        auto put = [&](const std::vector<int>& v) {
            size_t off = all.size();
            all.insert(all.end(), v.begin(), v.end());
            return off;
        };
        put(sj);
        put(si0);
        put(si1);
        h->off_cta_seg = put(cta);
        h->off_persist = put(persist);
        h->off_cta_slot = put(cta_slot);
        h->off_slot_blk = put(slot_blk);
        h->off_red_ptr = put(red_ptr);
        h->off_red_slot = put(red_slot);
        h->off_cta_item = put(gitems.cta_item);
        h->off_item_lo = put(gitems.lo);
        h->off_item_hi = put(gitems.hi);
        h->off_item_kind = put(gitems.kind);
        all.push_back(0);
        LPVS_CU(c, cudaMalloc(&h->seg_buf, sizeof(int) * all.size()));
        LPVS_CU(c, cudaMemcpyAsync(h->seg_buf, all.data(), sizeof(int) * all.size(), cudaMemcpyHostToDevice, c->st));
        LPVS_CU(c, cudaStreamSynchronize(c->st));
        LPVS_CU(c, cudaMalloc(&h->ypart, sizeof(double) * (size_t)slot_blk.size() * 128));
        }
    return LPVS_OK;
}

// Factor (G + I/mu), invert, allocate loop state.  d_G: Np x Np lower tiles (consumed), d_q: Np.
int admm_finish_create(lpvs_ctx* c, lpvs_admm* h, double* d_G, const double* d_q, const double* d_x0) {
    const int Np = h->Np, nb = Np / TB;
    const long long NN = (long long)Np * Np;
    h->M = d_G;  // owned by the handle from here on (freed by admm_release on any failure)
    // M = (G + I/mu)^-1 in place of G
    double* Y = nullptr;
    if (cudaMalloc(&Y, sizeof(double) * NN) != cudaSuccess) {
        cudaGetLastError();
        return fail(c, LPVS_E_NOMEM, "out of device memory (inverse workspace %lld MB)", (long long)(NN * 8 >> 20));
    }
    CholArgs ca{};
    ca.G = d_G;
    ca.strideG = NN;
    ca.Y = Y;
    ca.strideY = NN;
    ca.Linv = ws<double>(c, BUF_LINV, (size_t)nb * TB * TB);
    ca.strideLinv = (long long)nb * TB * TB;
    ca.info = ws<int>(c, BUF_INFO, 1);
    ca.Np = Np;
    ca.nb = nb;
    if (!ca.Linv || !ca.info) {
        cudaFree(Y);
        return fail(c, LPVS_E_NOMEM, "out of device memory (factor workspace)");
    }
    cudaMemsetAsync(ca.info, 0, sizeof(int), c->st);
    launch_diag_prepare(d_G, NN, Np, h->ncc, h->zero_first, nullptr, 1.0 / h->mu, 1, c->st);
    c->launches += 1 + potrf(ca, 1, c->sms, c->st, &c->la);
    int pinfo = 0;
    cudaMemcpyAsync(&pinfo, ca.info, sizeof(int), cudaMemcpyDeviceToHost, c->st);
    cudaError_t e = cudaStreamSynchronize(c->st);
    if (e != cudaSuccess) {
        cudaFree(Y);
        return fail(c, LPVS_E_CUDA, "factorisation failed: %s", cudaGetErrorString(e));
    }
    if (pinfo) {
        cudaFree(Y);
        return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown of (G + I/mu) at internal pivot %d", pinfo);
    }
    c->launches += potri(ca, 1, c->st);
    if (cudaMalloc(&h->vecs, sizeof(double) * 7 * Np) != cudaSuccess) {
        cudaStreamSynchronize(c->st);
        cudaFree(Y);
        return fail(c, LPVS_E_NOMEM, "out of memory");
    }
    double* q = h->vecs;
    const bool permuted = !h->h_order.empty();
    if (permuted) {
        // group prox: bring M and q into ADMM order (groups contiguous); the inverse workspace becomes M
        bool ok = cudaMalloc(&h->d_order, sizeof(int) * Np) == cudaSuccess &&
                  cudaMalloc(&h->d_pos, sizeof(int) * Np) == cudaSuccess;
        if (!ok) {
            cudaStreamSynchronize(c->st);
            cudaFree(Y);
            return fail(c, LPVS_E_NOMEM, "out of memory");
        }
        std::vector<int> pos((size_t)Np);
        for (int p = 0; p < Np; p++) pos[h->h_order[p]] = p;
        cudaMemcpyAsync(h->d_order, h->h_order.data(), sizeof(int) * Np, cudaMemcpyHostToDevice, c->st);
        cudaMemcpyAsync(h->d_pos, pos.data(), sizeof(int) * Np, cudaMemcpyHostToDevice, c->st);
        k_permute_sym<<<dim3((Np + 255) / 256, Np), 256, 0, c->st>>>(d_G, Y, h->d_order, Np);
        k_permute_vec<<<(Np + 255) / 256, 256, 0, c->st>>>(d_q, q, h->d_order, Np);
        c->launches += 2;
        e = cudaStreamSynchronize(c->st);
        h->M = Y;
        cudaFree(d_G);
    } else {
        cudaMemcpyAsync(q, d_q, sizeof(double) * Np, cudaMemcpyDeviceToDevice, c->st);
        e = cudaStreamSynchronize(c->st);
        cudaFree(Y);
    }
    if (e != cudaSuccess) return fail(c, LPVS_E_CUDA, "inverse failed: %s", cudaGetErrorString(e));
    // cooperative grid: one CTA per SM, never more CTAs than rows/2
    int maxb = 0;
    int grid = std::min(c->sms, std::max(1, Np / 8));
    int rows_max = (Np + grid - 1) / grid;
    size_t smem = admm_smem(Np, rows_max + 1);
    if (smem > 220 * 1024) return fail(c, LPVS_E_UNSUPPORTED, "ADMM problem too large for the resident rhs (Np=%d)", Np);
    LPVS_CU(c, cudaFuncSetAttribute(k_admm<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    LPVS_CU(c, cudaFuncSetAttribute(k_admm<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    LPVS_CU(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&maxb, k_admm<true>, ADMM_THREADS, smem));
    if (maxb < 1) return fail(c, LPVS_E_UNSUPPORTED, "ADMM kernel does not fit on an SM");
    h->grid = grid;
    // variant: SYMV over the lower triangle when M cannot live in L2 (or when forced), else GEMV over full M
    const bool big = 8.0 * Np * (double)Np > 96.0 * 1024 * 1024;
    h->symv = c->admm_symv < 0 ? (big && Np <= 24576) : (c->admm_symv != 0);
    GroupItems gitems;
    if (h->symv) {
        gitems = build_group_items(h, c->sms);
        h->max_item = gitems.max_item;
        size_t sm2 = admm_smem_symv(Np, h->max_item);
        if (sm2 > 220 * 1024) {
            if (c->admm_symv > 0) return fail(c, LPVS_E_UNSUPPORTED, "ADMM SYMV variant: Np=%d too large", Np);
            h->symv = 0;  // the GEMV variant only needs the resident rhs
        }
    }
    if (h->symv) {
        size_t sm2 = admm_smem_symv(Np, h->max_item);
        LPVS_CU(c, cudaFuncSetAttribute(k_admm_symv<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm2));
        LPVS_CU(c, cudaFuncSetAttribute(k_admm_symv<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm2));
        h->grid = grid = c->sms;
        if (c->admm_m32) {
            // Float32 callers (SURVEY 8f n2): the inverse is stored in single precision -- half the bytes every iteration
            // streams -- and accumulated in double; the double copy is released
            if (cudaMalloc(&h->M32, sizeof(float) * NN) != cudaSuccess) {
                cudaGetLastError();
                return fail(c, LPVS_E_NOMEM, "out of device memory (single-precision inverse)");
            }
            k_to_float<<<(unsigned)((NN + 255) / 256), 256, 0, c->st>>>(h->M, h->M32, NN);
            c->launches++;
            LPVS_CU(c, cudaStreamSynchronize(c->st));
            cudaFree(h->M);
            h->M = nullptr;
        }
        int rcp = build_symv_plan(c, h, gitems, 0, (long long)nb * (nb + 1) / 2);
        if (rcp) return rcp;
    }
    LPVS_CU(c, cudaMalloc(&h->part, sizeof(double) * 2 * grid));
    LPVS_CU(c, cudaMalloc(&h->d_iters, sizeof(long long)));
    LPVS_CU(c, cudaMalloc(&h->d_res, sizeof(double)));
    LPVS_CU(c, cudaMalloc(&h->d_flags, sizeof(int) * 2));
    LPVS_CU(c, cudaEventCreate(&h->e0));
    LPVS_CU(c, cudaEventCreate(&h->e1));
    if (permuted && d_x0) return fail(c, LPVS_E_UNSUPPORTED, "start vector with a group prox");
    k_admm_init<<<(Np + 255) / 256, 256, 0, c->st>>>(q, d_x0, Np, h->mu, h->quad, h->vecs + Np, h->vecs + 2 * Np,
                                                    h->vecs + 3 * Np, h->vecs + 5 * Np);
    c->launches++;
    h->rbuf = 0;
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    return LPVS_OK;
}

}  // namespace lpvs

extern "C" {

int lpvs_admm_run(lpvs_admm* h, int64_t max_iters, double tol, int64_t* iters_done, double* residual,
                  int* converged) {
    if (!h) return LPVS_E_BAD_ARG;
    lpvs_ctx* c = h->ctx;
    Lock lk(c->mu);
    cudaSetDevice(c->device);
    if (iters_done) *iters_done = 0;
    if (max_iters <= 0 || h->converged) {
        if (residual) *residual = h->residual;
        if (converged) *converged = h->converged;
        return LPVS_OK;
    }
    const int Np = h->Np;
    AdmmArgs a{};
    a.M = h->M;
    a.M32 = h->M32;
    a.Np = Np;
    a.q = h->vecs;
    a.x = h->vecs + Np;
    a.z = h->vecs + 2 * Np;
    a.u = h->vecs + 3 * Np;
    a.v = h->vecs + 4 * Np;
    a.r = h->vecs + 5 * Np;
    a.mu = h->mu;
    a.quad = h->quad;
    a.prox = h->prox;
    a.pparam = h->pparam;
    a.ref_half = h->half;
    a.zero_first = h->zero_first;
    a.goff = h->goff;
    a.gmem = h->gmem;
    a.ngroups = h->ngroups;
    a.part = h->part;
    a.max_iters = max_iters;
    a.tol = tol;
    a.check_every = c->admm_check_every;
    a.rbuf0 = h->rbuf;
    a.iters_out = h->d_iters;
    a.res_out = h->d_res;
    a.conv_out = h->d_flags;
    a.rbuf_out = h->d_flags + 1;
    // clock-stamp trace of a few iterations (tools/admm_trace.py): a developer build only (-DLPVS_ADMM_TRACE_HOOK); the
    // production library neither reads the environment nor writes files
    struct TraceBuf {
        long long* p = nullptr;
        ~TraceBuf() { if (p) cudaFree(p); }  // freed on every exit path
    } trace_buf;
    long long*& d_trace = trace_buf.p;
    const char* trace_path = nullptr;
#ifdef LPVS_ADMM_TRACE_HOOK
    trace_path = getenv("LPVS_ADMM_TRACE");
#endif
    if (trace_path && *trace_path && max_iters > 16) {
        LPVS_CU(c, cudaMalloc(&d_trace, sizeof(long long) * TRACE_ITERS * h->grid * 8));
        LPVS_CU(c, cudaMemsetAsync(d_trace, 0, sizeof(long long) * TRACE_ITERS * h->grid * 8, c->st));
        a.trace = d_trace;
        a.trace_it0 = max_iters / 2;
    }
    LPVS_CU(c, cudaEventRecord(h->e0, c->st));
    if (h->shard_world > 1) {
        if (!h->shard_connected) return fail(c, LPVS_E_BAD_ARG, "sharded ADMM handle is not connected to its peers");
        SymvPlan sp{};
        sp.seg_j = h->seg_buf;
        sp.seg_i0 = h->seg_buf + h->nseg;
        sp.seg_i1 = h->seg_buf + 2 * h->nseg;
        sp.cta_seg = h->seg_buf + h->off_cta_seg;
        sp.cta_persist = h->seg_buf + h->off_persist;
        sp.cta_slot = h->seg_buf + h->off_cta_slot;
        sp.slot_blk = h->seg_buf + h->off_slot_blk;
        sp.red_ptr = h->seg_buf + h->off_red_ptr;
        sp.red_slot = h->seg_buf + h->off_red_slot;
        sp.cta_item = h->seg_buf + h->off_cta_item;
        sp.item_lo = h->seg_buf + h->off_item_lo;
        sp.item_hi = h->seg_buf + h->off_item_hi;
        sp.item_kind = h->seg_buf + h->off_item_kind;
        sp.ypart = h->ypart;
        ShardArgs sh{};
        sh.rank = h->shard_rank;
        sh.world = h->shard_world;
        for (int k = 0; k <= h->shard_world; k++) sh.rb[k] = h->shard_rb[k];
        for (int k = 0; k < h->shard_world; k++) sh.base[k] = h->peer_base[k];
        sh.off_recv = h->off_recv;
        sh.off_rhs = h->off_rhs;
        sh.off_resid = h->off_resid;
        sh.off_flagA = h->off_flagA;
        sh.off_flagB = h->off_flagB;
        sh.off_abort = h->off_abort;
        sh.off_cnt = h->off_cnt;
        sh.off_resid2 = h->off_resid2;
        sh.off_recv2 = h->off_recv2;
        sh.v2 = h->grid <= SHARD_MAXGRID ? c->shard_exchange : 0;
        sh.rows_max = h->shard_rows_max;
        sh.it_base = h->iters_total;
        sh.spin_limit = 6000000000LL;  // ~3 s of SM clocks: a peer that is this late is gone
        void* args[] = {&a, &sp, &sh};
        if ((h->prox == LPVS_PROX_GROUP_L2 || h->prox == LPVS_PROX_BALL_L0) && sh.v2 != 2)
            return fail(c, LPVS_E_UNSUPPORTED, "sharded group prox / IndBallL0 need LPVS_OPT_SHARD_EXCHANGE = 2 on every rank");
        LPVS_CU(c, cudaLaunchCooperativeKernel((void*)k_admm_symv_sharded, dim3(h->grid), dim3(ADMM_THREADS), args,
                                               admm_smem_symv(Np, h->max_item), c->st));
        const int own0 = h->shard_rb[h->shard_rank] * 128;
        const int ownn = (h->shard_rb[h->shard_rank + 1] - h->shard_rb[h->shard_rank]) * 128;
        k_shard_broadcast<<<(ownn + 255) / 256, 256, 0, c->st>>>(a.x, a.z, a.u, own0, ownn, Np, sh, h->off_xzu);
        c->launches++;
    } else if (h->symv) {
        SymvPlan sp{};
        sp.seg_j = h->seg_buf;
        sp.seg_i0 = h->seg_buf + h->nseg;
        sp.seg_i1 = h->seg_buf + 2 * h->nseg;
        sp.cta_seg = h->seg_buf + h->off_cta_seg;
        sp.cta_persist = h->seg_buf + h->off_persist;
        sp.cta_slot = h->seg_buf + h->off_cta_slot;
        sp.slot_blk = h->seg_buf + h->off_slot_blk;
        sp.red_ptr = h->seg_buf + h->off_red_ptr;
        sp.red_slot = h->seg_buf + h->off_red_slot;
        sp.cta_item = h->seg_buf + h->off_cta_item;
        sp.item_lo = h->seg_buf + h->off_item_lo;
        sp.item_hi = h->seg_buf + h->off_item_hi;
        sp.item_kind = h->seg_buf + h->off_item_kind;
        sp.ypart = h->ypart;
        void* args[] = {&a, &sp};
        LPVS_CU(c, cudaLaunchCooperativeKernel(h->M32 ? (void*)k_admm_symv<float> : (void*)k_admm_symv<double>, dim3(h->grid),
                                               dim3(ADMM_THREADS), args, admm_smem_symv(Np, h->max_item), c->st));
    } else {
        int rows_max = (Np + h->grid - 1) / h->grid;
        size_t smem = admm_smem(Np, rows_max + 1);
        void* args[] = {&a};
        const bool stream = 8.0 * Np * (double)Np > 96.0 * 1024 * 1024;  // M larger than what L2 can keep
        void* kfn = stream ? (void*)k_admm<true> : (void*)k_admm<false>;
        LPVS_CU(c, cudaLaunchCooperativeKernel(kfn, dim3(h->grid), dim3(ADMM_THREADS), args, smem, c->st));
    }
    LPVS_CU(c, cudaEventRecord(h->e1, c->st));
    c->launches++;
    long long its = 0;
    double res = 0.0;
    int flags[2] = {0, 0};
    LPVS_CU(c, cudaMemcpyAsync(&its, h->d_iters, sizeof(long long), cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaMemcpyAsync(&res, h->d_res, sizeof(double), cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaMemcpyAsync(flags, h->d_flags, sizeof(int) * 2, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    if (d_trace) {
        std::vector<long long> tr((size_t)TRACE_ITERS * h->grid * 8);
        cudaMemcpy(tr.data(), d_trace, sizeof(long long) * tr.size(), cudaMemcpyDeviceToHost);
        if (FILE* fp = fopen(trace_path, "wb")) {
            int hdr[2] = {TRACE_ITERS, h->grid};
            fwrite(hdr, sizeof(int), 2, fp);
            fwrite(tr.data(), sizeof(long long), tr.size(), fp);
            fclose(fp);
        }
    }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->e0, h->e1);
    h->last_ms = ms;
    h->last_iters = its;
    h->iters_total += its;
    h->residual = res;
    if (flags[0] < 0)
        return fail(c, LPVS_E_CUDA, "sharded ADMM: a peer GPU did not answer within the spin budget (loop aborted)");
    h->converged = flags[0];
    h->rbuf = flags[1];
    if (iters_done) *iters_done = its;
    if (residual) *residual = res;
    if (converged) *converged = flags[0];
    return LPVS_OK;
}

int lpvs_admm_shard_begin(lpvs_admm* h, int rank, int world) {
    if (!h) return LPVS_E_BAD_ARG;
    lpvs_ctx* c = h->ctx;
    Lock lk(c->mu);
    cudaSetDevice(c->device);
    const int Np = h->Np, nb = Np / TB;
    if (world < 2 || world > SHARD_MAXP || rank < 0 || rank >= world)
        return fail(c, LPVS_E_BAD_ARG, "sharded ADMM: world must be 2..%d and 0 <= rank < world", SHARD_MAXP);
    if (h->M32) return fail(c, LPVS_E_UNSUPPORTED, "sharded ADMM: not with the single-precision inverse (LPVS_OPT_ADMM_M32)");
    // element-wise prox operators with every exchange; the group prox (ls_sparse_spectral_lpv, BASELINE configs[3]) with
    // exchange 2, where every rank holds every row after the all-reduce and groups cannot straddle ranks
    const bool group = h->prox == LPVS_PROX_GROUP_L2 && c->shard_exchange == 2;
    const bool ball = h->prox == LPVS_PROX_BALL_L0 && c->shard_exchange == 2;  // redundant selection on every rank
    if (h->prox != LPVS_PROX_L1 && h->prox != LPVS_PROX_L0 && !group && !ball)
        return fail(c, LPVS_E_UNSUPPORTED,
                    "sharded ADMM supports NormL1 / NormL0, and the group prox / IndBallL0 with LPVS_OPT_SHARD_EXCHANGE = 2");
    if ((!h->h_order.empty() && !group) || nb < world || h->shard_world > 1 || h->iters_total > 0)
        return fail(c, LPVS_E_UNSUPPORTED, "sharded ADMM: needs a fresh problem with at least `world` 128-blocks");
    h->symv = 1;
    h->grid = c->sms;
    GroupItems gitems = build_group_items(h, c->sms);  // empty unless the prox is the group one
    h->max_item = gitems.max_item;
    if (admm_smem_symv(Np, h->max_item) > 220 * 1024)
        return fail(c, LPVS_E_UNSUPPORTED, "sharded ADMM: Np=%d too large", Np);
    LPVS_CU(c, cudaFuncSetAttribute(k_admm_symv_sharded, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)admm_smem_symv(Np, h->max_item)));
    // this rank's contiguous share of the lower-triangle blocks, and the 128-row blocks every rank owns
    const long long T = (long long)nb * (nb + 1) / 2;
    int rc = build_symv_plan(c, h, gitems, T * rank / world, T * (rank + 1) / world);
    if (rc) return rc;
    cudaFree(h->part);
    h->part = nullptr;
    LPVS_CU(c, cudaMalloc(&h->part, sizeof(double) * 2 * h->grid));
    h->shard_rows_max = 0;
    for (int k = 0; k <= world; k++) h->shard_rb[k] = (int)((long long)nb * k / world);
    for (int k = 0; k < world; k++) h->shard_rows_max = std::max(h->shard_rows_max, (h->shard_rb[k + 1] - h->shard_rb[k]) * 128);
    long long off = 0;
    h->off_recv = off;   off += (long long)world * h->shard_rows_max;
    h->off_rhs = off;    off += 2LL * Np;
    h->off_resid = off;  off += 2LL * SHARD_MAXP;
    h->off_flagA = off;  off += SHARD_MAXP;
    h->off_flagB = off;  off += SHARD_MAXP;
    h->off_abort = off;  off += 4;
    h->off_cnt = off;    off += 2;
    h->off_resid2 = off; off += 2LL * SHARD_MAXP * SHARD_MAXGRID;
    h->off_recv2 = off;  off += 2LL * world * Np;
    h->off_xzu = off;    off += 3LL * Np;
    LPVS_CU(c, cudaMalloc(&h->xchg, sizeof(double) * off));
    LPVS_CU(c, cudaMemsetAsync(h->xchg, 0, sizeof(double) * off, c->st));
    // the current right-hand side (rhs of iteration 0) moves into the exchange region, buffer 0
    LPVS_CU(c, cudaMemcpyAsync(h->xchg + h->off_rhs, h->vecs + 5 * Np + (long long)h->rbuf * Np, sizeof(double) * Np,
                               cudaMemcpyDeviceToDevice, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    h->rbuf = 0;
    h->shard_rank = rank;
    h->shard_world = world;
    h->shard_connected = 0;
    for (int k = 0; k < SHARD_MAXP; k++) h->peer_base[k] = nullptr;
    h->peer_base[rank] = h->xchg;
    return LPVS_OK;
}

int lpvs_admm_shard_handle(lpvs_admm* h, void* handle64) {
    if (!h || !handle64 || h->shard_world < 2) return LPVS_E_BAD_ARG;
    lpvs_ctx* c = h->ctx;
    Lock lk(c->mu);
    cudaSetDevice(c->device);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t mh;
    LPVS_CU(c, cudaIpcGetMemHandle(&mh, h->xchg));
    memcpy(handle64, &mh, 64);
    return LPVS_OK;
}

int lpvs_admm_shard_connect(lpvs_admm* h, const void* handles) {
    if (!h || !handles || h->shard_world < 2) return LPVS_E_BAD_ARG;
    lpvs_ctx* c = h->ctx;
    Lock lk(c->mu);
    cudaSetDevice(c->device);
    for (int k = 0; k < h->shard_world; k++) {
        if (k == h->shard_rank) continue;
        cudaIpcMemHandle_t mh;
        memcpy(&mh, (const char*)handles + 64 * k, 64);
        void* p = nullptr;
        LPVS_CU(c, cudaIpcOpenMemHandle(&p, mh, cudaIpcMemLazyEnablePeerAccess));
        h->peer_base[k] = (double*)p;
    }
    h->shard_connected = 1;
    return LPVS_OK;
}

int lpvs_admm_size(const lpvs_admm* h) { return h ? h->nref : 0; }

int lpvs_prox_fourier(lpvs_ctx* c, int prox_kind, double prox_param, double gamma, const double* v, int Nf,
                      int zero_first, double* z) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    cudaSetDevice(c->device);
    if (!v || !z || Nf <= 0 || !(gamma > 0.0)) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (prox_kind < LPVS_PROX_L1 || prox_kind > LPVS_PROX_BALL_L0)
        return fail(c, LPVS_E_BAD_ARG, "prox kind %d not valid for the Fourier layout", prox_kind);
    zero_first = zero_first ? 1 : 0;
    const int nref = 2 * Nf - zero_first, Np = (Nf + FB - 1) / FB * TB;
    double* d_ref;
    int rc;
    if ((rc = upload(c, BUF_MISC, v, nref, &d_ref))) return rc;
    double* w = ws<double>(c, BUF_X, (size_t)7 * Np + nref);  // v, x, u, z, q, rn, (unused), out
    if (!w) return fail(c, LPVS_E_NOMEM, "out of device memory");
    LPVS_CU(c, cudaMemsetAsync(w, 0, sizeof(double) * (7 * (size_t)Np + nref), c->st));
    launch_scatter_ref_vec(c, d_ref, Nf, zero_first, nref, Np, w);
    LPVS_CU(c, cudaMemcpyAsync(w + Np, w, sizeof(double) * Np, cudaMemcpyDeviceToDevice, c->st));  // x = v, u = 0
    AdmmArgs a{};
    a.Np = Np;
    a.v = w;
    a.x = w + Np;
    a.u = w + 2 * Np;
    a.z = w + 3 * Np;
    a.q = w + 4 * Np;
    a.mu = gamma;
    a.prox = prox_kind;
    a.pparam = prox_param;
    a.ref_half = Nf;
    a.zero_first = zero_first;
    k_prox_only<<<1, ADMM_THREADS, 0, c->st>>>(a, w + 5 * Np);
    k_gather_vec<<<(nref + 255) / 256, 256, 0, c->st>>>(a.z, nref, Nf, zero_first, nullptr, w + 7 * Np);
    c->launches += 2;
    LPVS_CU(c, cudaMemcpyAsync(z, w + 7 * Np, sizeof(double) * nref, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    return inputs_finite(c);
}

int lpvs_admm_get(lpvs_admm* h, double* x, double* z) {
    if (!h) return LPVS_E_BAD_ARG;
    lpvs_ctx* c = h->ctx;
    Lock lk(c->mu);
    cudaSetDevice(c->device);
    double* tmp = ws<double>(c, BUF_X, (size_t)2 * h->nref);
    if (!tmp) return fail(c, LPVS_E_NOMEM, "out of device memory");
    const int Np = h->Np;
    // sharded handles: every owner broadcast its rows of x, z, u into each rank's exchange region after the run
    const double* xsrc = h->shard_world > 1 ? h->xchg + h->off_xzu : h->vecs + Np;
    const double* zsrc = h->shard_world > 1 ? h->xchg + h->off_xzu + Np : h->vecs + 2 * Np;
    k_gather_vec<<<(h->nref + 255) / 256, 256, 0, c->st>>>(xsrc, h->nref, h->half, h->zero_first, h->d_pos, tmp);
    k_gather_vec<<<(h->nref + 255) / 256, 256, 0, c->st>>>(zsrc, h->nref, h->half, h->zero_first, h->d_pos,
                                                           tmp + h->nref);
    c->launches += 2;
    if (x) LPVS_CU(c, cudaMemcpyAsync(x, tmp, sizeof(double) * h->nref, cudaMemcpyDeviceToHost, c->st));
    if (z) LPVS_CU(c, cudaMemcpyAsync(z, tmp + h->nref, sizeof(double) * h->nref, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    if (h->kind == 1) {
        // reference order of the LPV ADMM vector is the group-permuted one (src/lasso.jl:47-50):
        // position p = f*2Nvv + k  <->  un-permuted f + k*Nf, k = 0..2Nvv-1 over [Re | Im] columns
        const int Nf = h->lpv_nf, n2 = h->nref;
        std::vector<double> t((size_t)n2);
        for (double* vec : {x, z}) {
            if (!vec) continue;
            for (int j = 0; j < n2; j++) {
                int f = j % Nf, k = j / Nf;
                t[(size_t)f * (n2 / Nf) + k] = vec[j];
            }
            std::copy(t.begin(), t.end(), vec);
        }
    }
    return LPVS_OK;
}

int lpvs_admm_result(lpvs_admm* h, double* out) {
    if (!h || !out) return LPVS_E_BAD_ARG;
    lpvs_ctx* c = h->ctx;
    Lock lk(c->mu);
    cudaSetDevice(c->device);
    // complex column cc -> (z_re, z_im); Fourier zero frequency has no imaginary coefficient
    const int Np = h->Np, ncx = h->half;
    double* tmp = ws<double>(c, BUF_X, (size_t)2 * h->nref + 2);
    if (!tmp) return fail(c, LPVS_E_NOMEM, "out of device memory");
    k_gather_vec<<<(h->nref + 255) / 256, 256, 0, c->st>>>(
        h->shard_world > 1 ? h->xchg + h->off_xzu + Np : h->vecs + 2 * Np, h->nref, h->half, h->zero_first, h->d_pos, tmp);
    c->launches++;
    std::vector<double> z((size_t)h->nref);
    LPVS_CU(c, cudaMemcpyAsync(z.data(), tmp, sizeof(double) * h->nref, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    for (int k = 0; k < ncx; k++) {
        out[2 * k] = z[k];
        int j = ncx + k - h->zero_first;
        out[2 * k + 1] = (h->zero_first && k == 0) ? 0.0 : z[j];
    }
    return LPVS_OK;
}

int lpvs_admm_last_timing(const lpvs_admm* h, double* ms, double* bytes_per_iter) {
    if (!h) return LPVS_E_BAD_ARG;
    if (ms) *ms = h->last_ms;
    if (bytes_per_iter) {
        // algorithmic bytes of the variant actually run: full M (GEMV) or the lower-triangle blocks (SYMV)
        double nb = h->Np / 128.0;
        *bytes_per_iter = h->symv ? nb * (nb + 1.0) / 2.0 * 128.0 * 128.0 * (h->M32 ? 4.0 : 8.0)
                                  : 8.0 * (double)h->Np * (double)h->Np;
    }
    return LPVS_OK;
}

void lpvs_admm_free(lpvs_admm* h) {
    if (!h) return;
    lpvs_ctx* c = h->ctx;
    Lock lk(c->mu);
    admm_release(h);
}

}  // extern "C"

namespace lpvs {
lpvs_admm* admm_new(lpvs_ctx* c) {
    lpvs_admm* h = new lpvs_admm();
    h->ctx = c;
    c->live_admm.push_back(h);
    return h;
}
void admm_release_all(lpvs_ctx* c) {
    while (!c->live_admm.empty()) admm_release(c->live_admm.back());
}
void admm_delete(lpvs_admm* h) { admm_release(h); }
void admm_set_problem(lpvs_admm* h, int kind, int Np, int ncc, int zero_first, int nref, int half, int prox,
                      double pparam, double mu, int quad, int lpv_nf, int lpv_nvv) {
    h->kind = kind;
    h->Np = Np;
    h->ncc = ncc;
    h->zero_first = zero_first;
    h->nref = nref;
    h->half = half;
    h->prox = prox;
    h->pparam = pparam;
    h->mu = mu;
    h->quad = quad;
    h->lpv_nf = lpv_nf;
    h->lpv_nvv = lpv_nvv;
}
int admm_set_groups(lpvs_ctx* c, lpvs_admm* h, const std::vector<int>& goff, const std::vector<int>& gmem) {
    // gmem lists the internal index of every member, group after group, then the entries outside every group:
    // that IS the ADMM order.  The loop vectors and M are permuted into it (admm_finish_create), so on the device
    // the groups are the contiguous ranges goff[g]..goff[g+1] and the member table is the identity.
    h->ngroups = (int)goff.size() - 2;
    if ((int)gmem.size() != h->Np) return fail(c, LPVS_E_BAD_ARG, "group table does not cover the vector");
    h->h_order = gmem;
    h->h_goff = goff;
    std::vector<int> ident(gmem.size());
    for (size_t k = 0; k < ident.size(); k++) ident[k] = (int)k;
    LPVS_CU(c, cudaMalloc(&h->goff, sizeof(int) * goff.size()));
    LPVS_CU(c, cudaMalloc(&h->gmem, sizeof(int) * std::max<size_t>(1, ident.size())));
    LPVS_CU(c, cudaMemcpyAsync(h->goff, goff.data(), sizeof(int) * goff.size(), cudaMemcpyHostToDevice, c->st));
    LPVS_CU(c, cudaMemcpyAsync(h->gmem, ident.data(), sizeof(int) * ident.size(), cudaMemcpyHostToDevice, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    return LPVS_OK;
}
}  // namespace lpvs
