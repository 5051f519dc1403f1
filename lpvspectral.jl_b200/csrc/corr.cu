// LPVS_PHASE_STRUCTURED_REF: the structured Gram matrix (structured.cu) made parity-grade.
//
// The trigonometric sums give G0 = A0' W A0 for the IDEAL phases theta_ks = 2 pi (f0 + k df) t_s; the reference evaluates its
// basis at phi_ks = fl(fl(2 pi f_k) t_s) (src/lsfft.jl:34,41).  The difference eps_ks = phi_ks - theta_ks (<= 6e-9 rad at
// BASELINE cfg5a) is per-element rounding noise, not a function of i +- j, so it does not fit the Toeplitz + Hankel structure --
// but it is tiny, and to first order (the eps^2 terms are < 1e-17)
//     G_ref = G0 + D'B + B'D,     b_ref = b0 + D'y,     B = A0 (cos, -sin),  D = diag(W) (dA/dphi o eps) = W eps (-sin, -cos).
// dG is 1e-10 of G and is needed to ~3 digits: a HALF-PRECISION tensor-core GEMM (mma.sync m16n8k16, f16 operands, f32
// accumulation).  eps is taken exactly in FP64 -- the rounding error of the product by one FMA, w t - fl(w t), plus
// (fl(2 pi f_k) - 2 pi f_k) t -- scaled by a power of two and rounded to f16.
//
// FP64 instructions stall behind HMMA bursts on this SM (ncu, profiles/r02_summary.md: `math pipe throttle` on the first DMUL of
// every synthesis phase), so the FP64 part runs ONCE per (column, sample) in a table pass and the GEMM kernel is FP64-free:
//   k_corr_max      max |t|, max |W| of the sample range -> the power-of-two scales (computed identically by every kernel)
//   k_corr_tables   per (8-column chain group, sample): eps S as 8 halves (16 B), the group's anchor (cos, -sin) of the
//                   reference phase (float2), per sample the step rotation e^{-i 2 pi df t} (float2); Wf = float(W wsc)
//   k_gram_corr     one CTA per (lower 128 x 128 tile, problem), warp-specialised: 8 producer warps turn table entries into f16
//                   operand panels (FP32 angle-addition chain from the anchor), 8 consumer warps run the MMAs; G += scale * acc
//   k_rhs_corr      one CTA per (64-frequency block, problem): b += D'[y u], eps in FP64 (21 bits), products / sums in FP32
// 3 bytes of table per (column, sample), window-independent (overlapping windows and all tiles of a window share them).
//
// Accuracy (tests/test_gpu_structured.py, tools/corr_emulation.py): dG to 3e-4 of itself; cfg5a window 4166 (phase 2.6e7 rad,
// cond(A) 2e5): 4e-9 -> 5e-11 against the reference-literal N-rhs LU solve on the CPU.
#include <cuda_fp16.h>

#include "gram.cuh"

namespace lpvs {

namespace {

constexpr int LDH = 72;            // smem row stride in halves: 64 k' + 8 pad = 144 B, conflict-free ldmatrix and STS.32
constexpr int PANEL_H = TB * LDH;  // halves per panel buffer
constexpr int LDM = TB + 1;        // row stride of the FP32 accumulator tile the epilogue stages in shared memory
constexpr double CF = 6755399441055744.0;  // 1.5 * 2^52: x + CF has round(x) in its low word (|x| < 2^31)

// powers of two of one sample range: S with |eps| S <= 2^21 for every element (the table keeps eps S 2^-7 <= 2^14 as f16), wsc with
// max|W| wsc < 1 (so |D| < 2^14 in f16), and the magic constant / shift that leave the fraction of a phase in turns in the
// low word of a double
struct CorrScales {
    double S, wsc, unscale;  // unscale = 1 / (S 2^-7 wsc)
    double cq;               // 1.5 * 2^(52 - fb): q + cq has frac(q) 2^fb in its low word
    int shl;                 // 32 - fb
};

__device__ __forceinline__ int exp_above(double x) {  // x < 2^result (x >= 0; zero / denormal -> -1022)
    return ((__double2hiint(x) >> 20) & 0x7ff) - 1022;
}
__device__ __forceinline__ double pow2i(int e) { return __hiloint2double((1023 + e) << 20, 0); }  // |e| <= 1022

__device__ __forceinline__ CorrScales corr_scales(const CorrArgs& a) {
    const double tm = a.scal[0], wm = a.scal[1];  // max |t|, max |W| (k_corr_max)
    CorrScales sc;
    // |w t - fl(w t)| <= |w t| 2^-53, |dw t| <= dwmax tmax
    const double epsmax = a.wmax * tm * 1.1102230246251565e-16 + a.dwmax * tm;
    const int sexp = min(21 - exp_above(epsmax), 600), wexp = min(-exp_above(wm), 600);
    sc.S = pow2i(sexp);
    sc.wsc = pow2i(wexp);
    sc.unscale = pow2i(7 - sexp) * pow2i(-wexp);
    const int tb = exp_above(a.wmax * tm * 0.15915494309189535);  // |phase| < 2^tb turns
    const int fb = max(1, min(24, 51 - tb));
    sc.cq = 1.5 * pow2i(52 - fb);
    sc.shl = 32 - fb;
    return sc;
}

// scal[0] = max |t_s| over [s0, s0 + ns), scal[1] = max |W_i| over [w0, w0 + nw) (1 without weights); non-negative doubles order
// like their bit patterns
__global__ void k_corr_max(const double* __restrict__ t, long long s0, long long ns, const double* __restrict__ W, long long w0,
                           long long nw, unsigned long long* __restrict__ scal) {
    double tm = 0.0, wm = W ? 0.0 : 1.0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < ns; i += stride) tm = fmax(tm, fabs(t[s0 + i]));
    if (W)
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += stride) wm = fmax(wm, fabs(W[w0 + i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        tm = fmax(tm, __shfl_xor_sync(0xffffffffu, tm, o));
        wm = fmax(wm, __shfl_xor_sync(0xffffffffu, wm, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(scal, (unsigned long long)__double_as_longlong(tm));
        atomicMax(scal + 1, (unsigned long long)__double_as_longlong(wm));
    }
}

// (cos, -sin)(2 pi q) in FP32 for a phase of q turns given as a double (|q| < 2^(51 - fb))
__device__ __forceinline__ float2 cis_turns_f32(double q_plus_cq, int shl) {
    const int fr = (int)((unsigned)__double2loint(q_plus_cq) << shl);  // frac(q) 2^32, signed: [-1/2, 1/2) turns
    const float ang = __int2float_rn(fr) * 1.4629180792671596e-9f;  // 2 pi / 2^32
    return make_float2(__cosf(ang), -__sinf(ang));
}

// grid (ceil(ns / 256), groups): thread = one sample of one 8-column chain group
__global__ void __launch_bounds__(256) k_corr_tables(const __grid_constant__ CorrArgs a) {
    const long long si = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (si >= a.tbl_ns) return;
    const int g = blockIdx.y;
    const CorrScales sc = corr_scales(a);
    const double t = a.t[a.tbl_base + si];
    const double negS = -sc.S;
    float ef[GRP];
    double p0 = 0.0;
#pragma unroll
    for (int j = 0; j < GRP; j++) {
        const double2 wj = a.wtab[g * GRP + j];      // (w, dw); zero beyond ncc
        const double p = __dmul_rn(wj.x, t);         // fl(w t)
        const double e = __fma_rn(wj.x, t, -p);      // w t - fl(w t), exact
        const double q = __fma_rn(e, negS, CF);      // fixed point: -(w t - p) S
        const int ei = __double2loint(__fma_rn(wj.y * sc.S, t, q));  // + (w - w_ideal) S t  =  eps S,  |.| <= 2^21
        ef[j] = (__int_as_float(0x4B400000 + ei) - 12582912.0f) * 0.0078125f;  // int -> float (exact below 2^22), 2^-7
        if (j == 0) p0 = p;
    }
    uint4 pk;
    __half2 h;
    h = __floats2half2_rn(ef[0], ef[1]);
    pk.x = *reinterpret_cast<unsigned*>(&h);
    h = __floats2half2_rn(ef[2], ef[3]);
    pk.y = *reinterpret_cast<unsigned*>(&h);
    h = __floats2half2_rn(ef[4], ef[5]);
    pk.z = *reinterpret_cast<unsigned*>(&h);
    h = __floats2half2_rn(ef[6], ef[7]);
    pk.w = *reinterpret_cast<unsigned*>(&h);
    a.eps[(long long)g * a.tbl_ns + si] = pk;
    a.anc[(long long)g * a.tbl_ns + si] = cis_turns_f32(__fma_rn(p0, 0.15915494309189535, sc.cq), sc.shl);  // reference phase
    if (g == 0) a.step[si] = cis_turns_f32(__fma_rn(a.df, t, sc.cq), sc.shl);
}

// Wf[i] = float(W[w0 + i] wsc)  (wsc alone without weights)
__global__ void k_corr_weights(const __grid_constant__ CorrArgs a, long long w0, long long nw) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nw) return;
    const CorrScales sc = corr_scales(a);
    a.wf[i] = (float)((a.W ? a.W[w0 + i] : 1.0) * sc.wsc);
}

// The 8 consecutive columns (one chain group) of one sample from their table entries: emit(j, Bc, Bs, Dc, Ds) with
// B = (cos, -sin) of the phase (FP32 angle-addition chain from the group's anchor) and D = W eps (-sin, -cos), scaled.  Columns
// beyond ncc have eps = 0, so their D is zero; their B is not (the consumers of G / b skip those rows and columns).
template <class Emit>
__device__ __forceinline__ void corr_group(const uint4& eps, float2 z, float wf, float2 step, Emit&& emit) {
    const unsigned w[4] = {eps.x, eps.y, eps.z, eps.w};
#pragma unroll
    for (int j = 0; j < GRP; j++) {
        const __half2 h = *reinterpret_cast<const __half2*>(&w[j >> 1]);
        const float de = ((j & 1) ? __high2float(h) : __low2float(h)) * wf;
        emit(j, z.x, z.y, de * z.y, -de * z.x);
        z = make_float2(fmaf(z.x, step.x, -z.y * step.y), fmaf(z.x, step.y, z.y * step.x));
    }
}

__device__ __forceinline__ void ldsm_x4(unsigned (&r)[4], const __half* p) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(s));
}
__device__ __forceinline__ void hmma16816(float (&c)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// table entries of one sample of a chunk for the chain groups gI (and gJ)
struct Entry {
    uint4 eI, eJ;
    float2 aI, aJ, step;
    float wf;
};

template <bool TWO>
__device__ __forceinline__ Entry load_entry(const CorrArgs& a, long long s_begin, int c, int lane, int gI, int gJ) {
    const int idx = c * KC + lane;
    const bool valid = idx < a.n && s_begin + idx < a.s_end;
    long long s = s_begin + idx;
    if (!valid) s = min(s_begin + (long long)a.n, a.s_end) - 1;
    const long long si = s - a.tbl_base;
    Entry e;
    e.eI = __ldg(a.eps + (long long)gI * a.tbl_ns + si);
    e.aI = __ldg(a.anc + (long long)gI * a.tbl_ns + si);
    if (TWO) {
        e.eJ = __ldg(a.eps + (long long)gJ * a.tbl_ns + si);
        e.aJ = __ldg(a.anc + (long long)gJ * a.tbl_ns + si);
    }
    e.step = __ldg(a.step + si);
    e.wf = valid ? __ldg(a.wf + (a.w_abs ? si : (s - s_begin))) : 0.f;
    return e;
}

constexpr int CORR_THREADS = 512;  // warps 0-7: MMA consumers (4 x 2, warp tile 32 x 64); warps 8-15: operand producers
constexpr int NSTAGE = 3;          // ring of operand panel pairs between producers and consumers
constexpr int STAGE_H = 2 * PANEL_H;  // halves per stage: P then Q
__device__ __forceinline__ void bar_consumers() { asm volatile("bar.sync 2, 256;\n" ::: "memory"); }

// Warp-specialised: the producers fill a ring of NSTAGE operand panel pairs, the consumers run the MMAs of a stage as soon as it
// is full and hand it back when their fragment loads are done (full / empty mbarriers): neither side waits for the other
// in lock-step.
// Off-diagonal tile (I > J): K' = 2 per sample, P = [D_I | B_I], Q = [B_J | D_J]  ->  acc = D_I'B_J + B_I'D_J.
// Diagonal tile: K' = 1 per sample, P = D_I, Q = B_I -> acc = M = D_I'B_I; the epilogue adds M + M'.
// full[s]: the 256 producer threads have written stage s; empty[s]: the 256 consumer threads have read it (mbarriers: arrive
// releases, the parity wait acquires)
template <bool DIAG>
__device__ __forceinline__ void produce_chunk(const Entry& cur, int c, int lane, __half* ring, int row0, uint64_t* full,
                                              uint64_t* empty) {
    const int st = c % NSTAGE;
    __half* P = ring + st * STAGE_H + row0 * LDH;
    __half* Q = P + PANEL_H;
    mbar_wait(empty + st, ((c / NSTAGE) + 1) & 1);  // first round: passes at once
    if (DIAG) {
        corr_group(cur.eI, cur.aI, cur.wf, cur.step, [&](int j, float bc, float bs, float dc, float ds) {
            P[j * LDH + lane] = __float2half_rn(dc);
            P[(j + FB) * LDH + lane] = __float2half_rn(ds);
            Q[j * LDH + lane] = __float2half_rn(bc);
            Q[(j + FB) * LDH + lane] = __float2half_rn(bs);
        });
    } else {
        corr_group(cur.eI, cur.aI, cur.wf, cur.step, [&](int j, float bc, float bs, float dc, float ds) {
            *reinterpret_cast<__half2*>(P + j * LDH + 2 * lane) = __floats2half2_rn(dc, bc);
            *reinterpret_cast<__half2*>(P + (j + FB) * LDH + 2 * lane) = __floats2half2_rn(ds, bs);
        });
        corr_group(cur.eJ, cur.aJ, cur.wf, cur.step, [&](int j, float bc, float bs, float dc, float ds) {
            *reinterpret_cast<__half2*>(Q + j * LDH + 2 * lane) = __floats2half2_rn(bc, dc);
            *reinterpret_cast<__half2*>(Q + (j + FB) * LDH + 2 * lane) = __floats2half2_rn(bs, ds);
        });
    }
    mbar_arrive(full + st);
}

// table entries run two chunks ahead of their use; the loop is unrolled by three so that the three entries in flight keep
// their registers (a rotating copy would wait for the newest load at the end of every chunk)
template <bool DIAG>
__device__ __forceinline__ void produce(const CorrArgs& a, long long s_begin, int nchunks, int lane, int gI, int gJ, __half* ring,
                                        int row0, uint64_t* full, uint64_t* empty) {
    const int last = nchunks - 1;
    Entry e0 = load_entry<!DIAG>(a, s_begin, 0, lane, gI, gJ);
    Entry e1 = load_entry<!DIAG>(a, s_begin, min(1, last), lane, gI, gJ);
    Entry e2;
    for (int c = 0; c < nchunks; c += 3) {
        e2 = load_entry<!DIAG>(a, s_begin, min(c + 2, last), lane, gI, gJ);
        produce_chunk<DIAG>(e0, c, lane, ring, row0, full, empty);
        if (c + 1 >= nchunks) break;
        e0 = load_entry<!DIAG>(a, s_begin, min(c + 3, last), lane, gI, gJ);
        produce_chunk<DIAG>(e1, c + 1, lane, ring, row0, full, empty);
        if (c + 2 >= nchunks) break;
        e1 = load_entry<!DIAG>(a, s_begin, min(c + 4, last), lane, gI, gJ);
        produce_chunk<DIAG>(e2, c + 2, lane, ring, row0, full, empty);
    }
}

// consumers: the MMAs of every chunk, warp tile 32 x 64 (A fragments from P, B fragments from Q)
template <bool DIAG>
__device__ __forceinline__ void consume(int nchunks, const __half* ring, int a_off, int b_off, uint64_t* full, uint64_t* empty,
                                        float (&acc)[2][8][4]) {
    constexpr int KS = DIAG ? KC / 16 : 2 * KC / 16;
    for (int c = 0; c < nchunks; c++) {
        const int st = c % NSTAGE;
        mbar_wait(full + st, (c / NSTAGE) & 1);
        const __half* P = ring + st * STAGE_H + a_off;
        const __half* Q = ring + st * STAGE_H + PANEL_H + b_off;
#pragma unroll
        for (int ks = 0; ks < KS; ks++) {
            unsigned af[2][4], bf[4][4];
#pragma unroll
            for (int i = 0; i < 2; i++) ldsm_x4(af[i], P + i * 16 * LDH + ks * 16);
#pragma unroll
            for (int jj = 0; jj < 4; jj++) ldsm_x4(bf[jj], Q + jj * 16 * LDH + ks * 16);
            if (ks == KS - 1) mbar_arrive(empty + st);  // this thread has read all it needs of the stage
#pragma unroll
            for (int jj = 0; jj < 4; jj++)
#pragma unroll
                for (int i = 0; i < 2; i++) {
                    hmma16816(acc[i][2 * jj], af[i], bf[jj][0], bf[jj][1]);
                    hmma16816(acc[i][2 * jj + 1], af[i], bf[jj][2], bf[jj][3]);
                }
        }
    }
}

__global__ void __launch_bounds__(CORR_THREADS, 1) k_gram_corr(const __grid_constant__ CorrArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __half* ring = reinterpret_cast<__half*>(smem_raw);  // [NSTAGE][P | Q][TB][LDH]: rows = functions of block I | block J
    uint64_t* full = reinterpret_cast<uint64_t*>(ring + NSTAGE * STAGE_H);
    uint64_t* empty = full + NSTAGE;
    if (threadIdx.x < 2 * NSTAGE) mbar_init(full + threadIdx.x, CORR_THREADS / 2);  // full[] and empty[] are contiguous
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    __syncthreads();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int I, J;
    tile_ij(blockIdx.x, I, J);
    const int prob = blockIdx.y;
    const long long s_begin = a.start0 + (long long)prob * a.hop;
    const bool diag = I == J;
    const int nchunks = (a.n + KC - 1) / KC;
    if (warp >= 8) {
        // ---- producers: warp = chain group (columns 8 g .. 8 g + 7 of a block), lane = sample of the chunk
        const int g = warp - 8;
        if (diag)
            produce<true>(a, s_begin, nchunks, lane, I * (FB / GRP) + g, 0, ring, GRP * g, full, empty);
        else
            produce<false>(a, s_begin, nchunks, lane, I * (FB / GRP) + g, J * (FB / GRP) + g, ring, GRP * g, full, empty);
    } else {
        // ---- consumers
        float acc[2][8][4];
#pragma unroll
        for (int i = 0; i < 2; i++)
#pragma unroll
            for (int j = 0; j < 8; j++)
#pragma unroll
                for (int q = 0; q < 4; q++) acc[i][j][q] = 0.f;
        // ldmatrix lane addresses: A = P rows (16 x 16: matrices (rows 0-7 | 8-15) x (k 0-7 | 8-15)), B = Q rows ((n 0-7 | 8-15) x k)
        const int wm = warp & 3, wn = warp >> 2, mi = lane >> 3;
        const int a_off = (wm * 32 + (mi & 1) * 8 + (lane & 7)) * LDH + (mi >> 1) * 8;
        const int b_off = (wn * 64 + (mi >> 1) * 8 + (lane & 7)) * LDH + (mi & 1) * 8;
        if (diag)
            consume<true>(nchunks, ring, a_off, b_off, full, empty, acc);
        else
            consume<false>(nchunks, ring, a_off, b_off, full, empty, acc);
        // the accumulators go through shared memory (over the panel buffers) so that all 16 warps write G, coalesced
        bar_consumers();  // every consumer is done with the panels
        float* sM = reinterpret_cast<float*>(smem_raw);
#pragma unroll
        for (int i = 0; i < 2; i++)
#pragma unroll
            for (int j = 0; j < 8; j++)
#pragma unroll
                for (int q = 0; q < 4; q++)
                    sM[(wm * 32 + i * 16 + (lane >> 2) + 8 * (q >> 1)) * LDM + wn * 64 + j * 8 + 2 * (lane & 3) + (q & 1)] =
                        acc[i][j][q];
    }
    __syncthreads();
    // G += gscale / (S wsc) * acc (diagonal tiles: M + M'); rows / columns of columns that do not exist (k >= ncc) stay as filled
    const float* sM = reinterpret_cast<const float*>(smem_raw);
    const int Np = a.nblk * TB;
    const double scl = a.gscale * corr_scales(a).unscale;
    double* Gt = a.G + (long long)prob * a.strideG + (long long)I * TB * Np + J * TB;
    const int cl = tid & (TB - 1);
    const bool cok = J * FB + (cl & (FB - 1)) < a.ncc;
    for (int r0 = 0; r0 < TB; r0 += 8 * (CORR_THREADS / TB)) {  // 8 rows per thread at a time: all loads, then all stores
        double gv[8];
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int rl = r0 + q * (CORR_THREADS / TB) + (tid >> 7);
            gv[q] = (cok && I * FB + (rl & (FB - 1)) < a.ncc) ? Gt[(long long)rl * Np + cl] : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int rl = r0 + q * (CORR_THREADS / TB) + (tid >> 7);
            float v = sM[rl * LDM + cl];
            if (diag) v += sM[cl * LDM + rl];
            if (cok && I * FB + (rl & (FB - 1)) < a.ncc) Gt[(long long)rl * Np + cl] = gv[q] + scl * (double)v;
        }
    }
}

// b += D'[y u]: thread = (sample of the chunk, chain group), FP32 accumulation over the chunks, fixed-order lane reduction.
// eps is taken in FP64 here (this kernel has no HMMAs to wait behind) and enters the products with 21 bits instead of the
// table's 11: b carries the residual of the correction at full weight (dx = G^-1 (db - dG x)), and with the f16 eps it was the
// larger of the two (8e-13 of b against 5e-14 of G at 2.6e7 rad).  Anchors, steps and weights still come from the tables.
struct RhsEntry {
    float2 anc, step;
    float wf, y0, y1;
    double t;
};
__device__ __forceinline__ RhsEntry load_rhs_entry(const CorrArgs& a, long long s_begin, int c, int lane, int g) {
    const int idx = c * KC + lane;
    const bool valid = idx < a.n && s_begin + idx < a.s_end;
    long long s = s_begin + idx;
    if (!valid) s = min(s_begin + (long long)a.n, a.s_end) - 1;  // weight 0 there
    const long long si = s - a.tbl_base;
    RhsEntry e;
    e.anc = __ldg(a.anc + (long long)g * a.tbl_ns + si);
    e.step = __ldg(a.step + si);
    e.wf = valid ? __ldg(a.wf + (a.w_abs ? si : (s - s_begin))) : 0.f;
    e.t = __ldg(a.t + s);
    e.y0 = (float)__ldg(a.y + s);
    e.y1 = a.nrhs > 1 ? (float)__ldg(a.u + s) : 0.f;
    return e;
}

__global__ void __launch_bounds__(NTHREADS) k_rhs_corr(const __grid_constant__ CorrArgs a) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int I = blockIdx.x, prob = blockIdx.y;
    const long long s_begin = a.start0 + (long long)prob * a.hop;
    const int g = I * (FB / GRP) + warp;
    const int kv = min(GRP, max(0, a.ncc - g * GRP));
    const int nchunks = (a.n + KC - 1) / KC;
    const CorrScales sc = corr_scales(a);
    const double negS = -sc.S;
    double2 wt[GRP];  // (w, dw S) of this warp's columns; zero beyond ncc
#pragma unroll
    for (int j = 0; j < GRP; j++) {
        wt[j] = a.wtab[g * GRP + j];
        wt[j].y *= sc.S;
    }
    float ac[2][GRP], as[2][GRP];
#pragma unroll
    for (int r = 0; r < 2; r++)
#pragma unroll
        for (int j = 0; j < GRP; j++) ac[r][j] = as[r][j] = 0.f;
    RhsEntry nxt = load_rhs_entry(a, s_begin, 0, lane, g);
    for (int c = 0; c < nchunks; c++) {
        const RhsEntry cur = nxt;
        nxt = load_rhs_entry(a, s_begin, c + 1 < nchunks ? c + 1 : c, lane, g);  // loads while this chunk is accumulated
        float2 z = cur.anc;
#pragma unroll
        for (int j = 0; j < GRP; j++) {
            const double p = __dmul_rn(wt[j].x, cur.t);       // fl(w t)
            const double e = __fma_rn(wt[j].x, cur.t, -p);    // w t - fl(w t), exact
            const double q = __fma_rn(e, negS, CF);
            const int ei = __double2loint(__fma_rn(wt[j].y, cur.t, q));  // eps S, |.| <= 2^21
            const float de = (__int_as_float(0x4B400000 + ei) - 12582912.0f) * 0.0078125f * cur.wf;  // the table's scaling
            const float dc = de * z.y, ds = -de * z.x;
            ac[0][j] = fmaf(dc, cur.y0, ac[0][j]);
            as[0][j] = fmaf(ds, cur.y0, as[0][j]);
            ac[1][j] = fmaf(dc, cur.y1, ac[1][j]);
            as[1][j] = fmaf(ds, cur.y1, as[1][j]);
            z = make_float2(fmaf(z.x, cur.step.x, -z.y * cur.step.y), fmaf(z.x, cur.step.y, z.y * cur.step.x));
        }
    }
    const int Np = a.nblk * TB;
    const double scl = a.bscale * sc.unscale;
    double* Bp = a.B + (long long)prob * a.strideB;
#pragma unroll
    for (int r = 0; r < 2; r++)
#pragma unroll
        for (int j = 0; j < GRP; j++) {
            float vc = ac[r][j], vs = as[r][j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                vc += __shfl_xor_sync(0xffffffffu, vc, o);
                vs += __shfl_xor_sync(0xffffffffu, vs, o);
            }
            if (lane == 0 && r < a.nrhs && j < kv) {
                double* b = Bp + (long long)r * Np + I * TB + GRP * warp + j;
                b[0] += scl * (double)vc;
                b[FB] += scl * (double)vs;
            }
        }
}

constexpr size_t CORR_SMEM = (size_t)NSTAGE * STAGE_H * sizeof(__half) + 2 * NSTAGE * sizeof(uint64_t);

}  // namespace

size_t corr_table_bytes_per_sample(int nblk) { return (size_t)nblk * (FB / GRP) * (sizeof(uint4) + sizeof(float2)) + sizeof(float2); }

// scales of the scale range, tables of the sample range [a.tbl_base, a.tbl_base + a.tbl_ns) (a.scal zeroed here); weights
// W[w0 .. w0 + nw) -> a.wf
int launch_corr_tables(const CorrArgs& a, long long w0, long long nw, cudaStream_t st) {
    cudaMemsetAsync(a.scal, 0, 2 * sizeof(double), st);
    k_corr_max<<<296, 256, 0, st>>>(a.t, a.scal_ns ? a.scal_base : a.tbl_base, a.scal_ns ? a.scal_ns : a.tbl_ns, a.W, w0, nw,
                                    reinterpret_cast<unsigned long long*>(a.scal));
    k_corr_tables<<<dim3((unsigned)((a.tbl_ns + 255) / 256), a.nblk * (FB / GRP)), 256, 0, st>>>(a);
    k_corr_weights<<<(unsigned)((nw + 255) / 256), 256, 0, st>>>(a, w0, nw);
    return 3;
}

int launch_gram_corr(const CorrArgs& a, int nproblems, cudaStream_t st) {
    static bool attr_done[64] = {};  // per device: function attributes belong to the device's context
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_done[dev & 63]) {
        cudaFuncSetAttribute(k_gram_corr, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CORR_SMEM);
        attr_done[dev & 63] = true;
    }
    int launched = 0;
    const int ntiles = a.nblk * (a.nblk + 1) / 2;
    for (int p0 = 0; p0 < nproblems; p0 += 32768) {
        const int np = nproblems - p0 < 32768 ? nproblems - p0 : 32768;
        CorrArgs b = a;
        b.start0 = a.start0 + (long long)p0 * a.hop;
        b.G = a.G + (long long)p0 * a.strideG;
        k_gram_corr<<<dim3(ntiles, np), CORR_THREADS, CORR_SMEM, st>>>(b);
        launched++;
    }
    return launched;
}

int launch_rhs_corr(const CorrArgs& a, int nproblems, cudaStream_t st) {
    int launched = 0;
    for (int p0 = 0; p0 < nproblems; p0 += 32768) {
        const int np = nproblems - p0 < 32768 ? nproblems - p0 : 32768;
        CorrArgs b = a;
        b.start0 = a.start0 + (long long)p0 * a.hop;
        b.B = a.B + (long long)p0 * a.strideB;
        k_rhs_corr<<<dim3(a.nblk, np), NTHREADS, 0, st>>>(b);
        launched++;
    }
    return launched;
}

// (w, dw) per complex column for the ideal grid f0 + k df: w = fl(2 pi f_k) as the reference forms it (src/lsfft.jl:34) and
// dw = w - 2 pi (f0 + k df) in double-double; also max |w| and max |dw| (the bounds the kernels scale eps by)
void structured_ref_wtab(double f0, double df, const double* f, int Nf, int ncol, double* out, double* wmax, double* dwmax) {
    const double P_HI = 6.283185307179586, P_LO = 2.4492935982947064e-16;
    *wmax = 0.0;
    *dwmax = 0.0;
    for (int k = 0; k < ncol; k++) out[2 * k] = out[2 * k + 1] = 0.0;
    for (int k = 0; k < Nf; k++) {
        const double w = P_HI * f[k];
        const double kd = (double)k * df, kd_lo = fma((double)k, df, -kd);
        const double s_hi = f0 + kd, bb = s_hi - f0;
        const double s_lo = ((f0 - (s_hi - bb)) + (kd - bb)) + kd_lo;
        const double ph = P_HI * s_hi, pe = fma(P_HI, s_hi, -ph);
        const double p_lo = fma(P_LO, s_hi, pe) + P_HI * s_lo;
        const double dw = (w - ph) - p_lo;
        out[2 * k] = w;
        out[2 * k + 1] = dw;
        if (fabs(w) > *wmax) *wmax = fabs(w);
        if (fabs(dw) > *dwmax) *dwmax = fabs(dw);
    }
}

}  // namespace lpvs
