// Fused basis synthesis -> DMMA SYRK.  See gram.cuh for the layout contract.
//
// Per CTA: one 128x128 tile (I,J), I >= J, of one problem's Gram; 8 warps as 4(M) x 2(N), warp tile 32x64,
// 64 FP64 accumulators per thread.  The k-dimension (samples) is consumed in chunks of 32: while the DMMAs run on
// the current chunk's smem tiles, the same threads synthesise the next chunk's tiles into the other buffer
// (software pipelined inside the k4-step loop because DMMA and DFMA share one pipe -- tools/fp64_probe.cu).
//
// GRAM_CHAIN synthesis (uniform frequency grid): thread (warp w, lane l) owns sample l of the chunk and the 8
// frequencies 64*blk+8w .. +7; it starts from an exact anchor e^{-i 2 pi f t} and advances with the per-sample
// rotation e^{-i 2 pi df t}: 4 FP64 ops per (cos,-sin) pair instead of ~35.  The anchor is the product of two table
// entries (double-double phases): one per (64-frequency block, sample) and one per (warp, sample) -- the block's first
// frequency turned by 8 w df -- so the table holds nblk + 8 rows per sample instead of 8 nblk.
#include "gram.cuh"

#include <stdlib.h>

#include <type_traits>

namespace lpvs {

namespace {

constexpr int STAGE_D = 2 * TILE_D;  // I tile, J tile (J = weighted copy)
#ifndef SYNTH_BURST
#define SYNTH_BURST 1
#endif
#ifndef GRAM_PAIR_SYNC
#define GRAM_PAIR_SYNC 0
#endif
constexpr int NSTAGE = 3;             // smem ring of the 8-warp kernel (per-stage mbarriers, no __syncthreads)

struct Pref {
    double2 aI, aJ, d;  // chain: anchors + step rotation
    double2 pw;         // chain: e^{-i 2 pi (8 w df) t}, folded into aI / aJ by resolve()
    double tt;          // direct: sample position
    long long si;       // table sample index
    double wt;
    double yv;   // rhs sample (diagonal tiles with the fused single right-hand side)
    bool valid;  // the weight is zeroed for invalid samples at the point of USE (no stall on the prefetch)
};

// GRAM_CHAINREF: z = e^{-i theta} with the exact phase theta = 2 pi (f_anchor + j df) t -> e^{-i phi}, phi = fl(w t) the
// reference's rounded phase.  phi - theta = dw t - (w t - fl(w t)); the product error is exact through one FMA, and the
// rotation by that angle (<= ~1e-8 rad) is first order: second-order terms are < 1e-16.  Pinned arithmetic (see above).
__device__ __forceinline__ double2 chain_ref_correct(double2 z, double2 wk, double t) {
    const double phr = __dmul_rn(wk.x, t);
    const double err = __fma_rn(wk.x, t, -phr);
    const double dlt = __fma_rn(wk.y, t, -err);
    return make_double2(__fma_rn(z.y, dlt, z.x), __fma_rn(-z.x, dlt, z.y));
}

template <int MODE, bool DIAG, bool RHS = false>
__device__ __forceinline__ Pref load_pref(const GramArgs& a, int c, long long s_begin, int lane, int w, int I,
                                          int J) {
    Pref p{};
    int idx = c * KC + lane;
    bool valid = idx < a.n && s_begin + idx < a.s_end;
    long long s = s_begin + idx;
    if (!valid) s = min(s_begin + (long long)a.n, a.s_end) - 1;
    int idc = (int)(s - s_begin);
    p.si = s - a.tbl_base;
    p.wt = 1.0;
    if (a.W) p.wt = a.W[a.w_abs ? s : (long long)idc];
    p.valid = valid;
    if (RHS) p.yv = a.y[s];
    if (gram_is_chain(MODE)) {
        p.aI = a.anc[(long long)I * a.tbl_ns + p.si];
        if (!DIAG) p.aJ = a.anc[(long long)J * a.tbl_ns + p.si];
        p.pw = a.anc[(long long)(a.nblk + w) * a.tbl_ns + p.si];
        p.d = a.del[p.si];
        if (MODE == GRAM_CHAINREF) p.tt = a.t[s];
    } else if (MODE == GRAM_DIRECT) {
        p.tt = a.t[s];
    }
    return p;
}

// value of complex column cc at the prefetched sample (slow paths)
template <int MODE>
__device__ __forceinline__ double2 synth_elem(const GramArgs& a, const Pref& p, int cc) {
    if (gram_is_chain(MODE)) return make_double2(0.0, 0.0);  // never taken: chain modes do not synthesise per element
    if (MODE == GRAM_DIRECT) {
        return cis_reference(a.f[cc], p.tt);
    } else {
        int fi = cc % a.lpv_nf, ki = cc / a.lpv_nf;
        double2 e = a.E[(long long)fi * a.tbl_ns + p.si];
        double k = a.Kt[(long long)ki * a.tbl_ns + p.si];
        return make_double2(e.x * k, e.y * k);
    }
}

// DIAG tiles (I == J) compute only the 20 of 32 pieces (16 rows x 32 columns) that touch the lower triangle: piece (r, c)
// is needed iff r >= 2c -- and of the four pieces that start ON the diagonal (r == 2c) only the left 16 columns, the right
// half lying strictly above it: 144 DMMAs per k4-step instead of 256.  The deal matters as much as the count.  (i) The two
// warps of an SM sub-partition (w and w+4) share one FP64 pipe and keep it busy only while BOTH have DMMAs to issue: a warp
// that finishes its chunk early waits at the stage barrier and leaves its partner to run alone.  (ii) A predicated-off DMMA
// still occupies the pipe (measured, profiles/r02_summary.md: a 36-DMMA deal with 4 of 40 predicated off ran exactly as
// long as the 40-DMMA deal and ncu counted 40), so every warp must execute the SAME instruction stream.  Hence: every warp
// takes two whole pieces that share their A or B fragments (16 DMMAs) plus 8 rows of one diagonal half piece (2 DMMAs; of
// the upper 8 rows the second is the one wasted 8x8 block): 18 per warp, 36 per sub-partition, no predicates.
//   w0 (7,0)(7,1)+(6,3)lo   w1 (6,0)(6,1)+(4,2)lo   w2 (5,0)(5,1)+(2,1)lo   w3 (6,2)(5,2)+(0,0)lo
//   w4 (7,2)(7,3)+(6,3)up   w5 (4,0)(4,1)+(4,2)up   w6 (3,0)(3,1)+(2,1)up   w7 (1,0)(2,0)+(0,0)up
// (History on cfg2, diagonal tiles alone: three lower 64x64 sub-blocks 48 per sub-partition; 40 with warp pairs 24 + 12:
// 24.6 ms at 71 % useful pipe time; 36 as 20 + 16 with predicates: 23.4 ms; this deal: see profiles/r02_summary.md.)
// RHS (diagonal tiles only, nrhs == 1): b_I = A_I' W y is accumulated by the threads that synthesise A_I anyway --
// 2 FMAs per synthesised element in the 16 accumulator registers the diagonal layout leaves free -- instead of a second
// pass over the anchor table (k_gram_rhs: 2.2 ms of a 85 ms step on cfg2).
template <int MODE, bool DIAG, bool RHS = false>
__device__ __forceinline__ void gram_tile(const GramArgs& a, int I, int J, int prob, double* smem) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int wm = w & 3, wn = w >> 2;
    const long long s_begin = a.start0 + (long long)prob * a.hop;
    const int nchunks = (a.n + KC - 1) / KC;
    // GRAM_CHAINREF: (w, dw) of the I block's and the J block's 64 complex columns, staged below
    const double2* sWtab = reinterpret_cast<const double2*>(smem + NSTAGE * STAGE_D + 8);

    double acc[4][8][2];   // off-diagonal: [i][j][e]; diagonal: viewed as [piece(3)][i(2)*4+j(4)][e(2)] = 48 used
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

    const int ccI0 = I * FB + w * GRP, ccJ0 = J * FB + w * GRP;
    const int rowc = (w * GRP) * LDT + lane;       // smem offset of the real-part row for j = 0
    const int rows = (FB + w * GRP) * LDT + lane;  // second-part row

    // masking is only needed when this warp's 8-column group is not entirely valid (warp-uniform)
    const bool maskI = ccI0 + GRP > a.ncc, maskJ = ccJ0 + GRP > a.ncc;
    const bool any_mask = maskI || (!DIAG && maskJ);
    // synthesise element j (of 8) of a chunk into stage buffer `st`.  CHAIN, off-diagonal: zJ is pre-scaled by the
    // sample weight (rotation is linear), so the J tile needs no per-element multiply.
    double rc[RHS ? GRP : 1], rs[RHS ? GRP : 1];
#pragma unroll
    for (int j = 0; j < (RHS ? GRP : 1); j++) rc[j] = rs[j] = 0.0;
    auto synth_step = [&](auto masked, const Pref& p, double2& zI, double2& zJ, int j, double* st) {
        double2 vI, vJ;
        if (MODE == GRAM_CHAIN) {
            vI = zI;
            vJ = DIAG ? make_double2(zI.x * p.wt, zI.y * p.wt) : zJ;
        } else if (MODE == GRAM_CHAINREF) {
            vI = chain_ref_correct(zI, sWtab[w * GRP + j], p.tt);
            vJ = DIAG ? make_double2(vI.x * p.wt, vI.y * p.wt) : chain_ref_correct(zJ, sWtab[FB + w * GRP + j], p.tt);
        } else {
            vI = synth_elem<MODE>(a, p, min(ccI0 + j, a.ncc - 1));
            vJ = DIAG ? vI : synth_elem<MODE>(a, p, min(ccJ0 + j, a.ncc - 1));
            vJ = make_double2(vJ.x * p.wt, vJ.y * p.wt);
        }
        if constexpr (decltype(masked)::value) {  // only the last (partial) 8-column group of a basis needs this
            if (maskI && ccI0 + j >= a.ncc) vI = make_double2(0.0, 0.0);
            if ((DIAG ? maskI : maskJ) && (DIAG ? ccI0 : ccJ0) + j >= a.ncc) vJ = make_double2(0.0, 0.0);
        }
        if (RHS) {  // p.yv already carries the (validity-resolved) weight
            rc[j] = fma(vI.x, p.yv, rc[j]);
            rs[j] = fma(vI.y, p.yv, rs[j]);
        }
        double* sI = st;
        double* sJ = st + TILE_D;
        sI[rowc + j * LDT] = vI.x;
        sI[rows + j * LDT] = vI.y;
        sJ[rowc + j * LDT] = vJ.x;
        sJ[rows + j * LDT] = vJ.y;
        if (gram_is_chain(MODE)) {
            zI = chain_rotate(zI, p.d);
            if (!DIAG) zJ = chain_rotate(zJ, p.d);
        }
    };
    auto chain_start_J = [&](const Pref& p) { return make_double2(p.aJ.x * p.wt, p.aJ.y * p.wt); };

    // prologue: chunk 0 into stage 0
    auto resolve = [](Pref& p) {
        p.wt = p.valid ? p.wt : 0.0;
        if (RHS) p.yv *= p.wt;
        if (gram_is_chain(MODE)) {  // anchor of this warp's 8-frequency group = block anchor x group power (pinned product)
            p.aI = chain_rotate(p.aI, p.pw);
            if (!DIAG) p.aJ = chain_rotate(p.aJ, p.pw);
        }
    };
    // 3-stage ring: full[s] completes when all 8 warps have stored their part of the chunk living in stage s.
    // A stage is rewritten two chunks after it was last read; passing full[] of the chunk in between proves every
    // warp has left that read, so no "empty" barrier is needed.
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + NSTAGE * STAGE_D);
    if (tid == 0) {
#pragma unroll
        for (int q = 0; q < NSTAGE; q++) mbar_init(&full[q], NTHREADS / 32);
    }
    if (MODE == GRAM_CHAINREF && tid < 2 * FB) {
        double2* dst = reinterpret_cast<double2*>(smem + NSTAGE * STAGE_D + 8);
        dst[tid] = a.wtab[(tid < FB ? I : J) * FB + (tid & (FB - 1))];
    }
    __syncthreads();
    // prologue: chunk 0 into stage 0
    Pref p1 = load_pref<MODE, DIAG, RHS>(a, 0, s_begin, lane, w, I, J);
    resolve(p1);
    {
        double2 zI = p1.aI, zJ = chain_start_J(p1);
#pragma unroll
        for (int j = 0; j < GRP; j++) synth_step(std::true_type{}, p1, zI, zJ, j, smem);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&full[0]);
    if (nchunks > 1) p1 = load_pref<MODE, DIAG, RHS>(a, 1, s_begin, lane, w, I, J);
    mbar_wait(&full[0], 0);

    // fragment bases: off-diagonal 32(M) x 64(N) warp tile; diagonal: per-piece offsets added below
    const int fragA = DIAG ? (lane >> 2) * LDT + (lane & 3) : (32 * wm + (lane >> 2)) * LDT + (lane & 3);
    const int fragB = DIAG ? (lane >> 2) * LDT + (lane & 3) : (64 * wn + (lane >> 2)) * LDT + (lane & 3);
    // diagonal tile: this warp's pieces (16-row strip pr, 32-column strip pc); the third piece of warps 0-3 shares
    // the A fragments of the first
    // nibble w of each constant = the value for warp w (table in the comment above gram_tile)
    const int pr0 = (0x13476567u >> (4 * w)) & 15, pc0 = (0x00022000u >> (4 * w)) & 15;
    const int pr1 = (0x23475567u >> (4 * w)) & 15, pc1 = (0x01132111u >> (4 * w)) & 15;
    const int prh = (0x02460246u >> (4 * w)) & 15, pch = (0x01230123u >> (4 * w)) & 15;
    const int ih = w < 4 ? 1 : 0;  // which 8 rows of the diagonal half piece (1 = lower)
    const int offA0 = 16 * pr0 * LDT, offA1 = 16 * pr1 * LDT, offAh = (16 * prh + 8 * ih) * LDT;
    const int offB0 = 32 * pc0 * LDT, offB1 = 32 * pc1 * LDT, offBh = 32 * pch * LDT;

    // staggering the bursts of an SMSP's two warps (kk = 0 / 4) measured no better: 78.0 vs 77.7 ms with the exact-phase
    // burst, SYNTH_BURST=3 re-measures it with the longer reference-phase burst (profiles/r02_summary.md)
    int st_cur = 0;
    // SYNTH_BURST == 4: the two warps of an SM sub-partition (w and w+4) burst half a chunk apart, with the burst position a
    // COMPILE-TIME constant of two specialised copies of the loop (a run-time position makes every unrolled k-step carry a
    // predicated copy of the burst: SYNTH_BURST == 3, measured slower)
    auto chunk_loop = [&](auto bk_tag) {
    constexpr int BKC = decltype(bk_tag)::value;
    const int burst_kk = SYNTH_BURST == 3 ? (w >> 2) * 4 : BKC;
    for (int c = 0; c < nchunks; c++) {
        const int st_nxt = st_cur == NSTAGE - 1 ? 0 : st_cur + 1;
        double* cur = smem + st_cur * STAGE_D;
        double* nxt = smem + st_nxt * STAGE_D;
        const bool have_next = (c + 1 < nchunks);
        Pref p2 = p1;
        if (c + 2 < nchunks) p2 = load_pref<MODE, DIAG, RHS>(a, c + 2, s_begin, lane, w, I, J);
        resolve(p1);  // p1 was loaded one iteration ago: no stall
        double2 zI = p1.aI, zJ = chain_start_J(p1);
        const double* pa = cur + fragA;
        const double* pb = cur + TILE_D + fragB;
#pragma unroll
        for (int kk = 0; kk < KC / 4; kk++) {
            if (have_next) {
                if (SYNTH_BURST == 2) {
                    // two half bursts (kk = 0 and kk = 4), published after the second
                    if (kk == 0 || kk == 4) {
                        const int j0 = kk == 0 ? 0 : GRP / 2;
                        if (any_mask) {
#pragma unroll
                            for (int j = 0; j < GRP / 2; j++) synth_step(std::true_type{}, p1, zI, zJ, j0 + j, nxt);
                        } else {
#pragma unroll
                            for (int j = 0; j < GRP / 2; j++) synth_step(std::false_type{}, p1, zI, zJ, j0 + j, nxt);
                        }
                    } else if (kk == 5) {
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&full[st_nxt]);
                    }
                } else if (SYNTH_BURST) {
                    // whole next chunk in one burst: fewer DMMA<->DFMA interleave points (79.1 -> 77.7 ms)
                    if (kk == burst_kk) {
#if GRAM_PAIR_SYNC == 1  // the two warps of an SM sub-partition start their bursts together (named barrier per pair)
                        asm volatile("bar.sync %0, 64;" ::"r"(1 + (w & 3)) : "memory");
#elif GRAM_PAIR_SYNC == 2  // all eight warps start their bursts together
                        asm volatile("bar.sync 1, 256;" ::: "memory");
#endif
                        if (any_mask) {  // warp-uniform: the masked variant costs 128 selects per chunk
#pragma unroll
                            for (int j = 0; j < GRP; j++) synth_step(std::true_type{}, p1, zI, zJ, j, nxt);
                        } else {
#pragma unroll
                            for (int j = 0; j < GRP; j++) synth_step(std::false_type{}, p1, zI, zJ, j, nxt);
                        }
                    } else if (kk == burst_kk + 1) {
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&full[st_nxt]);
                    }
                } else if (kk < GRP / 2) {  // the next chunk is synthesised in the first half of this one ...
                    synth_step(std::true_type{}, p1, zI, zJ, 2 * kk, nxt);
                    synth_step(std::true_type{}, p1, zI, zJ, 2 * kk + 1, nxt);
                } else if (kk == GRP / 2) {  // ... and published half a chunk before anyone needs it
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&full[st_nxt]);
                }
            }
            if (!DIAG) {
                mma_step(pa, pb, kk, acc);
            } else {
                // every fragment of the k-step is requested up front, in its own registers (the diagonal path holds 40
                // accumulators against the off-diagonal path's 64, so there is room): one exposed shared-memory latency per
                // k-step instead of one per piece.  Pieces that share a row / column strip simply load it twice.
                double fa0[2], fa1[2], fah, fb0[4], fb1[4], fbh[2];
#pragma unroll
                for (int i = 0; i < 2; i++) fa0[i] = pa[offA0 + 8 * i * LDT + 4 * kk];
#pragma unroll
                for (int j = 0; j < 4; j++) fb0[j] = pb[offB0 + 8 * j * LDT + 4 * kk];
#pragma unroll
                for (int i = 0; i < 2; i++) fa1[i] = pa[offA1 + 8 * i * LDT + 4 * kk];
#pragma unroll
                for (int j = 0; j < 4; j++) fb1[j] = pb[offB1 + 8 * j * LDT + 4 * kk];
                fah = pa[offAh + 4 * kk];  // 8 rows x left 16 columns of a piece that starts on the diagonal
#pragma unroll
                for (int j = 0; j < 2; j++) fbh[j] = pb[offBh + 8 * j * LDT + 4 * kk];
#pragma unroll
                for (int i = 0; i < 2; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) dmma884(acc[0][i * 4 + j][0], acc[0][i * 4 + j][1], fa0[i], fb0[j]);
#pragma unroll
                for (int i = 0; i < 2; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) dmma884(acc[1][i * 4 + j][0], acc[1][i * 4 + j][1], fa1[i], fb1[j]);
#pragma unroll
                for (int j = 0; j < 2; j++) dmma884(acc[2][j][0], acc[2][j][1], fah, fbh[j]);
            }
        }
        p1 = p2;
        if (have_next) mbar_wait(&full[st_nxt], ((c + 1) / NSTAGE) & 1);
        st_cur = st_nxt;
    }
    };
    if (SYNTH_BURST == 4 && w >= 4)
        chunk_loop(std::integral_constant<int, 4>{});
    else
        chunk_loop(std::integral_constant<int, 0>{});

    // epilogue
    const int Np = a.nblk * TB;
    double* Gp = a.G + (long long)prob * a.strideG;
    if (RHS) {
        double* Bp = a.B + (long long)prob * a.strideB;
#pragma unroll
        for (int j = 0; j < GRP; j++) {
            double vc = rc[j], vs = rs[j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                vc += __shfl_xor_sync(0xffffffffu, vc, o);
                vs += __shfl_xor_sync(0xffffffffu, vs, o);
            }
            if (lane == 0) {
                const bool ok = ccI0 + j < a.ncc;
                Bp[I * TB + w * GRP + j] = ok ? vc * a.bscale : 0.0;
                Bp[I * TB + FB + w * GRP + j] = ok ? vs * a.bscale : 0.0;
            }
        }
    }
    if (!DIAG) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            int row = I * TB + 32 * wm + 8 * i + (lane >> 2);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                int col = J * TB + 64 * wn + 8 * j + 2 * (lane & 3);
                double2 v = make_double2(acc[i][j][0] * a.gscale, acc[i][j][1] * a.gscale);
                *reinterpret_cast<double2*>(Gp + (long long)row * Np + col) = v;
            }
        }
    } else {
#pragma unroll
        for (int pz = 0; pz < 2; pz++) {
            const int pr = pz == 0 ? pr0 : pr1, pc = pz == 0 ? pc0 : pc1;
#pragma unroll
            for (int i = 0; i < 2; i++) {
                int row = I * TB + 16 * pr + 8 * i + (lane >> 2);
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    int col = I * TB + 32 * pc + 8 * j + 2 * (lane & 3);
                    double2 v = make_double2(acc[pz][i * 4 + j][0] * a.gscale, acc[pz][i * 4 + j][1] * a.gscale);
                    *reinterpret_cast<double2*>(Gp + (long long)row * Np + col) = v;
                }
            }
        }
        {  // 8 rows of a diagonal half piece; the 8x8 block right of the diagonal block's upper rows is not stored
            const int row = I * TB + 16 * prh + 8 * ih + (lane >> 2);
#pragma unroll
            for (int j = 0; j < 2; j++) {
                if (j > ih) break;
                const int col = I * TB + 32 * pch + 8 * j + 2 * (lane & 3);
                double2 v = make_double2(acc[2][j][0] * a.gscale, acc[2][j][1] * a.gscale);
                *reinterpret_cast<double2*>(Gp + (long long)row * Np + col) = v;
            }
        }
    }
}

// b = A' diag(W) [y u]: one CTA per (64-frequency block, problem); warp = chain group, lane = sample.
template <int MODE>
__global__ void __launch_bounds__(NTHREADS) k_gram_rhs(const __grid_constant__ GramArgs a) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int I = blockIdx.x, prob = blockIdx.y;
    const long long s_begin = a.start0 + (long long)prob * a.hop;
    const int nchunks = (a.n + KC - 1) / KC;
    const int cc0 = I * FB + w * GRP;
    double sc[2][GRP], ss[2][GRP];
#pragma unroll
    for (int r = 0; r < 2; r++)
#pragma unroll
        for (int j = 0; j < GRP; j++) sc[r][j] = ss[r][j] = 0.0;
    auto load_y = [&](const Pref& p, double& y0, double& y1) {  // raw loads; weights applied at use
        long long s = p.si + a.tbl_base;
        y0 = a.y ? a.y[s] : 0.0;
        y1 = (a.nrhs > 1 && a.u) ? a.u[s] : 0.0;
    };
    // two chunks of operands in flight per thread (the kernel is DRAM-latency bound: it streams the anchor table once)
    Pref pn = load_pref<MODE, true>(a, 0, s_begin, lane, w, I, I);
    double yn0, yn1;
    load_y(pn, yn0, yn1);
    Pref pm = pn;
    double ym0 = yn0, ym1 = yn1;
    if (nchunks > 1) {
        pm = load_pref<MODE, true>(a, 1, s_begin, lane, w, I, I);
        load_y(pm, ym0, ym1);
    }
    for (int c = 0; c < nchunks; c++) {
        const Pref p = pn;
        const double wte = p.valid ? p.wt : 0.0;
        const double y0 = yn0 * wte, y1 = yn1 * wte;
        pn = pm;
        yn0 = ym0;
        yn1 = ym1;
        if (c + 2 < nchunks) {
            pm = load_pref<MODE, true>(a, c + 2, s_begin, lane, w, I, I);
            load_y(pm, ym0, ym1);
        }
        double2 z = gram_is_chain(MODE) ? chain_rotate(p.aI, p.pw) : p.aI;
#pragma unroll
        for (int j = 0; j < GRP; j++) {
            double2 v = z;
            if (MODE == GRAM_CHAINREF) v = chain_ref_correct(z, a.wtab[cc0 + j], p.tt);
            if (!gram_is_chain(MODE)) v = (cc0 + j < a.ncc) ? synth_elem<MODE>(a, p, cc0 + j) : make_double2(0.0, 0.0);
            sc[0][j] = fma(v.x, y0, sc[0][j]);
            ss[0][j] = fma(v.y, y0, ss[0][j]);
            sc[1][j] = fma(v.x, y1, sc[1][j]);
            ss[1][j] = fma(v.y, y1, ss[1][j]);
            if (gram_is_chain(MODE)) z = chain_rotate(z, p.d);
        }
    }
    const int Np = a.nblk * TB;
    double* Bp = a.B + (long long)prob * a.strideB;
#pragma unroll
    for (int r = 0; r < 2; r++)
#pragma unroll
        for (int j = 0; j < GRP; j++) {
            double vc = sc[r][j], vs = ss[r][j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                vc += __shfl_xor_sync(0xffffffffu, vc, o);
                vs += __shfl_xor_sync(0xffffffffu, vs, o);
            }
            if (lane == 0 && r < a.nrhs) {
                bool ok = cc0 + j < a.ncc;
                Bp[(long long)r * Np + I * TB + w * GRP + j] = ok ? vc * a.bscale : 0.0;
                Bp[(long long)r * Np + I * TB + FB + w * GRP + j] = ok ? vs * a.bscale : 0.0;
            }
        }
}

// B[p][c] = A' diag(W) Y[:, c] for a chunk of RHS_MC channels: one CTA per (64-frequency block, problem, channel chunk),
// warp = chain group, lane = sample, as k_gram_rhs.  The columns are synthesised by the same helpers in the same pinned
// arithmetic, so they are bit-identical to the ones k_gram multiplies; every synthesised (cos, -sin) pair feeds all channels
// of the chunk.  FP64 FMA accumulation per lane, then the fixed-order shuffle reduction.
template <int MODE>
__global__ void __launch_bounds__(NTHREADS) k_gram_rhs_multi(const __grid_constant__ GramArgs a, const double* __restrict__ Y,
                                                             long long ldY, int C) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int I = blockIdx.x, prob = blockIdx.y, c0 = blockIdx.z * RHS_MC;
    const long long s_begin = a.start0 + (long long)prob * a.hop;
    const int nchunks = (a.n + KC - 1) / KC;
    const int cc0 = I * FB + w * GRP;
    const int nc = min(RHS_MC, C - c0);
    double sc[RHS_MC][GRP], ss[RHS_MC][GRP];
#pragma unroll
    for (int r = 0; r < RHS_MC; r++)
#pragma unroll
        for (int j = 0; j < GRP; j++) sc[r][j] = ss[r][j] = 0.0;
    auto load_y = [&](const Pref& p, double (&yv)[RHS_MC]) {  // raw loads; weights applied at use; absent channels read 0
        const long long s = p.si + a.tbl_base;
#pragma unroll
        for (int r = 0; r < RHS_MC; r++) yv[r] = r < nc ? Y[(long long)(c0 + r) * ldY + s] : 0.0;
    };
    // two chunks of operands in flight per thread, as k_gram_rhs
    Pref pn = load_pref<MODE, true>(a, 0, s_begin, lane, w, I, I);
    double yn[RHS_MC], ym[RHS_MC];
    load_y(pn, yn);
    Pref pm = pn;
#pragma unroll
    for (int r = 0; r < RHS_MC; r++) ym[r] = yn[r];
    if (nchunks > 1) {
        pm = load_pref<MODE, true>(a, 1, s_begin, lane, w, I, I);
        load_y(pm, ym);
    }
    for (int c = 0; c < nchunks; c++) {
        const Pref p = pn;
        const double wte = p.valid ? p.wt : 0.0;
        double yw[RHS_MC];
#pragma unroll
        for (int r = 0; r < RHS_MC; r++) {
            yw[r] = yn[r] * wte;
            yn[r] = ym[r];
        }
        pn = pm;
        if (c + 2 < nchunks) {
            pm = load_pref<MODE, true>(a, c + 2, s_begin, lane, w, I, I);
            load_y(pm, ym);
        }
        double2 z = gram_is_chain(MODE) ? chain_rotate(p.aI, p.pw) : p.aI;
#pragma unroll
        for (int j = 0; j < GRP; j++) {
            double2 v = z;
            if (MODE == GRAM_CHAINREF) v = chain_ref_correct(z, a.wtab[cc0 + j], p.tt);
            if (!gram_is_chain(MODE)) v = (cc0 + j < a.ncc) ? synth_elem<MODE>(a, p, cc0 + j) : make_double2(0.0, 0.0);
#pragma unroll
            for (int r = 0; r < RHS_MC; r++) {
                sc[r][j] = fma(v.x, yw[r], sc[r][j]);
                ss[r][j] = fma(v.y, yw[r], ss[r][j]);
            }
            if (gram_is_chain(MODE)) z = chain_rotate(z, p.d);
        }
    }
    const int Np = a.nblk * TB;
    double* Bp = a.B + (long long)prob * a.strideB;
#pragma unroll
    for (int r = 0; r < RHS_MC; r++)
#pragma unroll
        for (int j = 0; j < GRP; j++) {
            double vc = sc[r][j], vs = ss[r][j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                vc += __shfl_xor_sync(0xffffffffu, vc, o);
                vs += __shfl_xor_sync(0xffffffffu, vs, o);
            }
            if (lane == 0 && r < nc) {
                const bool ok = cc0 + j < a.ncc;
                Bp[(long long)(c0 + r) * Np + I * TB + w * GRP + j] = ok ? vc * a.bscale : 0.0;
                Bp[(long long)(c0 + r) * Np + I * TB + FB + w * GRP + j] = ok ? vs * a.bscale : 0.0;
            }
        }
}

template <int MODE>
__global__ void __launch_bounds__(NTHREADS, 1) k_gram(const __grid_constant__ GramArgs a) {
    extern __shared__ __align__(16) double smem[];
    int I, J;
    tile_ij(blockIdx.x, I, J);
#ifdef GRAM_DBG_SKIP  // timing experiments only (tools/build_variants.sh): 1 = skip diagonal tiles, 2 = skip the others
    if ((GRAM_DBG_SKIP == 1) == (I == J)) return;
#endif
    if (I == J) {
        if (a.fuse_rhs)
            gram_tile<MODE, true, true>(a, I, J, blockIdx.y, smem);
        else
            gram_tile<MODE, true, false>(a, I, J, blockIdx.y, smem);
    } else {
        gram_tile<MODE, false>(a, I, J, blockIdx.y, smem);
    }
}

// rows [0, nblk): e^{-i 2 pi f_{64 b} t_s} (the block's first frequency); rows [nblk, nblk + GRP): e^{-i 2 pi (8 j df) t_s}
// (the turn from the block's first frequency to the first frequency of chain group j; `pstep[j]` = fl(8 j df) is computed
// on the host so that the reference-phase table of make_fourier_plan describes exactly the frequency realised here);
// del[s] = e^{-i 2 pi df t_s}.  All phases are reduced in double-double turns.
struct PowSteps {
    double v[GRP];
};
__global__ void k_anchor_table(const double* __restrict__ t, long long s0, long long ns,
                               const double* __restrict__ f, int nblk, const __grid_constant__ PowSteps pstep, double df,
                               double2* __restrict__ anc, double2* __restrict__ del) {
    long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    int g = blockIdx.y;
    double tt = t[s0 + s];
    if (g == nblk + GRP) {
        del[s] = cis_turns_exact(df, tt);
    } else {
        const double fk = g < nblk ? f[g * FB] : pstep.v[g - nblk];
        anc[(long long)g * ns + s] = cis_turns_exact(fk, tt);
    }
}

__global__ void k_lpv_tables(const double* __restrict__ X, const double* __restrict__ V, long long N,
                             const double* __restrict__ w, int Nf, int Nvv, const double* __restrict__ centers,
                             double gamma, int coulomb, int normalize, double2* __restrict__ E,
                             double* __restrict__ Kt, int* __restrict__ nonfinite) {
    long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= N) return;
    double x = X[s], v = V[s];
    // E: exp(-i * fl(w_f * X_n))  (src/lsfft.jl:244: exp.(im*w.*X) then the trailing adjoint conjugates)
    for (int fi = 0; fi < Nf; fi++) E[(long long)fi * N + s] = cis_of_phase(__dmul_rn(w[fi], x));
    // K: exp(-gamma (v - c_k)^2) [* (sign v == sign c_k)] [/ sum]   (src/lsfft.jl:195-207)
    double sum = 0.0;
    double sv = (v > 0.0) - (v < 0.0);
    for (int k = 0; k < Nvv; k++) {
        double c = centers[k];
        double dv = v - c;
        double val = exp(-gamma * (dv * dv));
        if (coulomb) {
            double sc = (c > 0.0) - (c < 0.0);
            if (sv != sc) val = 0.0;
        }
        sum += val;
        Kt[(long long)k * N + s] = val;
    }
    if (normalize) {
        for (int k = 0; k < Nvv; k++) Kt[(long long)k * N + s] /= sum;
        // coulomb masks every basis function when sign(v) matches no centre (v == 0): 0/0, as in the reference
        // (src/lsfft.jl:199-207), which then returns NaNs; reported as LPVS_E_NONFINITE instead
        if (nonfinite && !(sum > 0.0 && isfinite(sum))) atomicOr(nonfinite, 2);
    }
}

}  // namespace

size_t gram_smem_bytes() { return NSTAGE * STAGE_D * sizeof(double) + 64 + 2 * FB * sizeof(double2); }

int launch_gram(int mode, const GramArgs& a, int nproblems, cudaStream_t st) {
    int launched = 0;
    static bool attr_done[64] = {};  // per device: function attributes belong to the device's context
    int dev = 0;
    cudaGetDevice(&dev);
    size_t smem = gram_smem_bytes();
    if (!attr_done[dev & 63]) {
        cudaFuncSetAttribute(k_gram<GRAM_CHAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_gram<GRAM_DIRECT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_gram<GRAM_LPV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_gram<GRAM_CHAINREF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_done[dev & 63] = true;
    }
    int ntiles = a.nblk * (a.nblk + 1) / 2;
    // gridDim.y is limited to 65535: launch in slabs
    for (int p0 = 0; p0 < nproblems; p0 += 32768) {
        int np = nproblems - p0 < 32768 ? nproblems - p0 : 32768;
        GramArgs b = a;
        b.start0 = a.start0 + (long long)p0 * a.hop;
        b.G = a.G + (long long)p0 * a.strideG;
        if (a.B) b.B = a.B + (long long)p0 * a.strideB;
        dim3 grid(ntiles, np);
        dim3 grid_rhs(a.nblk, np);
        // a single right-hand side rides along in the diagonal tiles; two need the separate pass
        b.fuse_rhs = (a.B && a.nrhs == 1 && a.y) ? 1 : 0;
        const bool rhs = a.B && a.nrhs > 0 && a.y && !b.fuse_rhs;
        if (mode == GRAM_CHAIN) {
            k_gram<GRAM_CHAIN><<<grid, NTHREADS, smem, st>>>(b);
            if (rhs) k_gram_rhs<GRAM_CHAIN><<<grid_rhs, NTHREADS, 0, st>>>(b);
        } else if (mode == GRAM_CHAINREF) {
            k_gram<GRAM_CHAINREF><<<grid, NTHREADS, smem, st>>>(b);
            if (rhs) k_gram_rhs<GRAM_CHAINREF><<<grid_rhs, NTHREADS, 0, st>>>(b);
        } else if (mode == GRAM_DIRECT) {
            k_gram<GRAM_DIRECT><<<grid, NTHREADS, smem, st>>>(b);
            if (rhs) k_gram_rhs<GRAM_DIRECT><<<grid_rhs, NTHREADS, 0, st>>>(b);
        } else {
            k_gram<GRAM_LPV><<<grid, NTHREADS, smem, st>>>(b);
            if (rhs) k_gram_rhs<GRAM_LPV><<<grid_rhs, NTHREADS, 0, st>>>(b);
        }
        launched += rhs ? 2 : 1;
    }
    return launched;
}

int launch_gram_rhs(int mode, const GramArgs& a, int nproblems, cudaStream_t st) {
    int launched = 0;
    for (int p0 = 0; p0 < nproblems; p0 += 32768) {
        int np = nproblems - p0 < 32768 ? nproblems - p0 : 32768;
        GramArgs b = a;
        b.start0 = a.start0 + (long long)p0 * a.hop;
        b.B = a.B + (long long)p0 * a.strideB;
        b.fuse_rhs = 0;
        dim3 grid_rhs(a.nblk, np);
        if (mode == GRAM_CHAIN)
            k_gram_rhs<GRAM_CHAIN><<<grid_rhs, NTHREADS, 0, st>>>(b);
        else if (mode == GRAM_CHAINREF)
            k_gram_rhs<GRAM_CHAINREF><<<grid_rhs, NTHREADS, 0, st>>>(b);
        else if (mode == GRAM_DIRECT)
            k_gram_rhs<GRAM_DIRECT><<<grid_rhs, NTHREADS, 0, st>>>(b);
        else
            k_gram_rhs<GRAM_LPV><<<grid_rhs, NTHREADS, 0, st>>>(b);
        launched++;
    }
    return launched;
}

int launch_gram_rhs_multi(int mode, const GramArgs& a, const double* Y, long long ldY, int C, int nproblems,
                          cudaStream_t st) {
    int launched = 0;
    for (int p0 = 0; p0 < nproblems; p0 += 32768) {
        int np = nproblems - p0 < 32768 ? nproblems - p0 : 32768;
        GramArgs b = a;
        b.start0 = a.start0 + (long long)p0 * a.hop;
        b.B = a.B + (long long)p0 * a.strideB;
        dim3 grid(a.nblk, np, (C + RHS_MC - 1) / RHS_MC);
        if (mode == GRAM_CHAIN)
            k_gram_rhs_multi<GRAM_CHAIN><<<grid, NTHREADS, 0, st>>>(b, Y, ldY, C);
        else if (mode == GRAM_CHAINREF)
            k_gram_rhs_multi<GRAM_CHAINREF><<<grid, NTHREADS, 0, st>>>(b, Y, ldY, C);
        else if (mode == GRAM_DIRECT)
            k_gram_rhs_multi<GRAM_DIRECT><<<grid, NTHREADS, 0, st>>>(b, Y, ldY, C);
        else
            k_gram_rhs_multi<GRAM_LPV><<<grid, NTHREADS, 0, st>>>(b, Y, ldY, C);
        launched++;
    }
    return launched;
}

void launch_anchor_table(const double* t, long long s0, long long ns, const double* f, int nblk, double df,
                         double2* anc, double2* del, cudaStream_t st) {
    PowSteps ps;
    for (int j = 0; j < GRP; j++) ps.v[j] = anchor_group_step(j, df);
    dim3 grid((unsigned)((ns + 255) / 256), nblk + GRP + 1);
    k_anchor_table<<<grid, 256, 0, st>>>(t, s0, ns, f, nblk, ps, df, anc, del);
}

void launch_lpv_tables(const double* X, const double* V, long long N, const double* w, int Nf, int Nvv,
                       const double* centers, double gamma, int coulomb, int normalize, double2* E, double* Kt,
                       int* nonfinite, cudaStream_t st) {
    k_lpv_tables<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(X, V, N, w, Nf, Nvv, centers, gamma, coulomb,
                                                              normalize, E, Kt, nonfinite);
}

}  // namespace lpvs
