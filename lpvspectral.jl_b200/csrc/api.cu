// C ABI of liblpvs.so (see include/lpvs.h): context, Fourier LS estimators, windowed estimators.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "ctx.h"

namespace lpvs {

int fail(lpvs_ctx* c, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    return code;
}

void* ws_raw(lpvs_ctx* c, int slot, size_t bytes) {
    DevBuf& b = c->buf[slot];
    if (bytes == 0) bytes = 16;
    if (b.cap < bytes) {
        if (b.p) {
            cudaStreamSynchronize(c->st);
            cudaFree(b.p);
        }
        b.p = nullptr;
        b.cap = 0;
        size_t want = bytes + bytes / 8;
        if (cudaMalloc(&b.p, want) != cudaSuccess) {
            cudaGetLastError();
            if (cudaMalloc(&b.p, bytes) != cudaSuccess) {
                cudaGetLastError();
                return nullptr;
            }
            want = bytes;
        }
        b.cap = want;
    }
    return b.p;
}

void gram_timer_reset(lpvs_ctx* c) {
    c->ev_used = 0;
    c->gram_ms = 0.0;
    c->gram_launches = 0;
    c->gram_flops = 0.0;
}
void gram_timer_begin(lpvs_ctx* c) {
    if ((int)c->ev.size() < c->ev_used + 2) {
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        c->ev.push_back(a);
        c->ev.push_back(b);
    }
    cudaEventRecord(c->ev[c->ev_used], c->st);
}
void gram_timer_end(lpvs_ctx* c, double flops, int launches) {
    cudaEventRecord(c->ev[c->ev_used + 1], c->st);
    c->ev_used += 2;
    c->gram_flops += flops;
    c->gram_launches += launches;
}
int gram_timer_resolve(lpvs_ctx* c) {
    double ms = 0.0;
    for (int i = 0; i < c->ev_used; i += 2) {
        float m = 0.f;
        if (cudaEventElapsedTime(&m, c->ev[i], c->ev[i + 1]) == cudaSuccess) ms += m;
    }
    c->gram_ms = ms;
    return 0;
}

int make_fourier_plan(lpvs_ctx* c, const double* f, int Nf, FourierPlan* pl) {
    if (!f || Nf <= 0) return fail(c, LPVS_E_BAD_ARG, "empty frequency vector");
    for (int k = 0; k < Nf; k++) {
        if (!isfinite(f[k])) return fail(c, LPVS_E_NONFINITE, "non-finite frequency at index %d", k);
        if (k > 0 && f[k] == 0.0)  // src/lsfft.jl:20-24
            return fail(c, LPVS_E_BAD_ARG, "If zero frequency is included it must be the first frequency");
    }
    pl->Nf = Nf;
    pl->zero_first = (f[0] == 0.0);
    pl->Nreg = 2 * Nf - pl->zero_first;
    pl->nblk = (Nf + FB - 1) / FB;
    pl->Np = pl->nblk * TB;
    pl->ngroups = anchor_rows(pl->nblk);  // rows of the chain anchor table
    pl->dd = 1.0 / sqrt(2.0 * (double)Nf);  // src/lsfft.jl:35
    pl->f0 = f[0];
    pl->df = Nf > 1 ? (f[Nf - 1] - f[0]) / (double)(Nf - 1) : 0.0;
    double fmaxabs = 0.0, dev = 0.0;
    for (int k = 0; k < Nf; k++) {
        fmaxabs = std::max(fmaxabs, fabs(f[k]));
        dev = std::max(dev, fabs(f[k] - (pl->f0 + k * pl->df)));
    }
    bool uniform = dev <= 8.0 * 2.220446049250313e-16 * fmaxabs;
    int mode = c->phase_mode;
    if (mode == LPVS_PHASE_AUTO) mode = uniform ? LPVS_PHASE_CHAIN_REF : LPVS_PHASE_DIRECT;
    if ((mode == LPVS_PHASE_CHAIN || mode == LPVS_PHASE_CHAIN_REF || mode == LPVS_PHASE_STRUCTURED ||
         mode == LPVS_PHASE_STRUCTURED_REF) && !uniform)
        return fail(c, LPVS_E_BAD_ARG,
                    "LPVS_PHASE_CHAIN / LPVS_PHASE_CHAIN_REF / LPVS_PHASE_STRUCTURED[_REF] require a uniformly spaced frequency grid");
    pl->structured_ref = mode == LPVS_PHASE_STRUCTURED_REF;
    pl->structured = mode == LPVS_PHASE_STRUCTURED || pl->structured_ref;
    // right-hand sides and operators (and windows re-done alone): the chains, with the phase class of the Gram matrices
    if (pl->structured) mode = pl->structured_ref ? LPVS_PHASE_CHAIN_REF : LPVS_PHASE_CHAIN;
    pl->mode = mode == LPVS_PHASE_CHAIN ? GRAM_CHAIN : (mode == LPVS_PHASE_CHAIN_REF ? GRAM_CHAINREF : GRAM_DIRECT);
    if (pl->structured) {  // table-row frequencies of the two-right-hand-side layout (a call with fewer uses a prefix)
        const StructuredLayout lay = structured_layout(pl->f0, Nf, 2);
        c->sfreq_host.assign((size_t)2 * lay.nrows, 0.0);
        structured_row_freqs(pl->f0, pl->df, Nf, 2, c->sfreq_host.data());
        double* d_sf = ws<double>(c, BUF_SFREQ, (size_t)2 * lay.nrows);
        if (!d_sf) return fail(c, LPVS_E_NOMEM, "out of device memory (sum-table frequencies)");
        LPVS_CU(c, cudaMemcpyAsync(d_sf, c->sfreq_host.data(), sizeof(double) * 2 * lay.nrows, cudaMemcpyHostToDevice, c->st));
        pl->d_sfreq = reinterpret_cast<const double2*>(d_sf);
    }
    if (pl->structured_ref) {  // (w, dw) against the ideal grid f0 + k df the sums realise
        const int ncol = pl->nblk * FB;
        c->cwtab_host.assign((size_t)2 * ncol, 0.0);
        structured_ref_wtab(pl->f0, pl->df, f, Nf, ncol, c->cwtab_host.data(), &pl->cw_max, &pl->cdw_max);
        double* d_cw = ws<double>(c, BUF_CWTAB, (size_t)2 * ncol);
        if (!d_cw) return fail(c, LPVS_E_NOMEM, "out of device memory (correction phase table)");
        LPVS_CU(c, cudaMemcpyAsync(d_cw, c->cwtab_host.data(), sizeof(double) * 2 * ncol, cudaMemcpyHostToDevice, c->st));
        pl->d_cwtab = reinterpret_cast<const double2*>(d_cw);
    }
    double* d_f = ws<double>(c, BUF_F, Nf);
    if (!d_f) return fail(c, LPVS_E_NOMEM, "out of device memory (f)");
    LPVS_CU(c, cudaMemcpyAsync(d_f, f, sizeof(double) * Nf, cudaMemcpyHostToDevice, c->st));
    pl->d_f = d_f;
    if (pl->mode == GRAM_CHAINREF) {
        // per column k = 64 b + 8 g + j: w = fl(2 pi f_k) (src/lsfft.jl:34) and dw = w - 2 pi (f_64b + fl(8 g df) + j df), the
        // difference between the reference's angular frequency and the one the chain realises (block anchor x group power,
        // then j steps of df: launch_anchor_table), in double-double
        const double P_HI = 6.283185307179586, P_LO = 2.4492935982947064e-16;
        const int ncol = pl->nblk * FB;
        c->wtab_host.assign((size_t)2 * ncol, 0.0);
        auto two_sum = [](double a, double b, double& lo) {
            const double s = a + b, bb = s - a;
            lo = (a - (s - bb)) + (b - bb);
            return s;
        };
        for (int k = 0; k < Nf; k++) {
            const int b64 = (k / FB) * FB, g = (k - b64) / GRP, j = k - b64 - g * GRP;
            const double w = P_HI * f[k];
            double e1, e2;
            const double a_hi = two_sum(f[b64], anchor_group_step(g, pl->df), e1);
            const double jd = (double)j * pl->df, jd_lo = fma((double)j, pl->df, -jd);
            const double s_hi = two_sum(a_hi, jd, e2);
            const double s_lo = (e1 + e2) + jd_lo;
            const double ph = P_HI * s_hi, pe = fma(P_HI, s_hi, -ph);
            const double pl_lo = fma(P_LO, s_hi, pe) + P_HI * s_lo;
            c->wtab_host[2 * k] = w;
            c->wtab_host[2 * k + 1] = (w - ph) - pl_lo;
        }
        double* d_w = ws<double>(c, BUF_WTAB, (size_t)2 * ncol);
        if (!d_w) return fail(c, LPVS_E_NOMEM, "out of device memory (phase table)");
        LPVS_CU(c, cudaMemcpyAsync(d_w, c->wtab_host.data(), sizeof(double) * 2 * ncol, cudaMemcpyHostToDevice, c->st));
        pl->d_wtab = reinterpret_cast<const double2*>(d_w);
    }
    return LPVS_OK;
}

// ---------------------------------------------------------------------------------------------------------
// small kernels: partial reduction, layout gathers, window accumulation
// ---------------------------------------------------------------------------------------------------------
__global__ void k_reduce_parts(double* __restrict__ out, const double* __restrict__ parts, long long count,
                               long long stride, int nparts, int accumulate) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    double s = accumulate ? out[i] : 0.0;
    for (int p = 0; p < nparts; p++) s += parts[(long long)p * stride + i];
    out[i] = s;
}

__global__ void k_check_finite(const double* __restrict__ v, long long n, int* flag) {
    bool bad = false;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        bad |= !isfinite(v[i]);
    if (bad) atomicOr(flag, 1);
}

// out[0] <- min(out[0], c) over the channels c (blockIdx.y) of Y holding a NaN / Inf
__global__ void k_first_nonfinite_channel(const double* __restrict__ Y, long long ldY, long long N, int* out) {
    const int ch = blockIdx.y;
    bool bad = false;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
        bad |= !isfinite(Y[ch * ldY + i]);
    if (bad) atomicMin(out, ch);
}

// out[0] = max(ridge, scale * maxdiag[0]): jitter ridge decided on the device
__global__ void k_jitter_ridge(const double* __restrict__ maxdiag, double ridge, double scale, double* __restrict__ out) {
    out[0] = fmax(ridge, scale * maxdiag[0]);
}

// Base.merge(yf, w::Windows2) (src/windows.jl:58-70): overlap-average of per-window outputs; one thread per sample, the
// covering windows added in window order (the reference's `ym[inds] .+= yf[i]` loop), then ./ max(count, 1)
__global__ void k_merge_windows(const double* __restrict__ pieces, long long K, int n, int hop, long long N,
                                double* __restrict__ out) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= N) return;
    long long k0 = s >= n ? (s - n + hop) / hop : 0;  // first window with k*hop + n > s
    long long k1 = s / hop;                           // last window with k*hop <= s
    if (k1 > K - 1) k1 = K - 1;
    double acc = 0.0;
    long long cnt = 0;
    for (long long k = k0; k <= k1; k++) {
        acc += pieces[k * n + (s - k * hop)];
        cnt++;
    }
    out[s] = acc / (double)(cnt > 0 ? cnt : 1);
}

// internal x ([nrhs][Np]) -> interleaved complex [nrhs][Nf]   (fourier2complex, src/utilities.jl:62-73)
__global__ void k_x_to_complex(const double* __restrict__ X, int Np, int Nf, int zero_first, int nrhs,
                               double* __restrict__ out) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= Nf) return;
    int pc = (k >> 6) * 128 + (k & 63);
    for (int r = 0; r < nrhs; r++) {
        double re = X[(long long)r * Np + pc];
        double im = (zero_first && k == 0) ? 0.0 : X[(long long)r * Np + pc + 64];
        out[((long long)r * Nf + k) * 2] = re;
        out[((long long)r * Nf + k) * 2 + 1] = im;
    }
}

// internal lower-tile G -> reference-ordered full symmetric Nreg x Nreg; internal b -> reference order
__device__ __forceinline__ int ref_to_internal(int j, int Nf, int zero_first) {
    if (j < Nf) return (j >> 6) * 128 + (j & 63);
    int k = j - Nf + zero_first;
    return (k >> 6) * 128 + 64 + (k & 63);
}
__global__ void k_gather_ref(const double* __restrict__ G, const double* __restrict__ B, int Np, int Nf,
                             int zero_first, int Nreg, double* __restrict__ Gout, double* __restrict__ bout) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    int i = blockIdx.y;
    if (j >= Nreg) return;
    int pi = ref_to_internal(i, Nf, zero_first), pj = ref_to_internal(j, Nf, zero_first);
    int a = max(pi, pj), b = min(pi, pj);
    double v = G[(long long)a * Np + b];  // always the lower element: bit-symmetric output
    Gout[(long long)i * Nreg + j] = v;
    if (bout && i == 0) bout[j] = B[pj];
}
__global__ void k_scatter_ref_vec(const double* __restrict__ xin, int Nf, int zero_first, int Nreg, int Np,
                                  double* __restrict__ xout) {
    // reference-ordered vector -> internal layout (dummies zero)
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= Np) return;
    int q = p >> 7, r = p & 127, part = r >> 6, cc = q * 64 + (r & 63);
    double v = 0.0;
    if (cc < Nf && !(zero_first && part == 1 && cc == 0)) {
        int j = part == 0 ? cc : (Nf + cc - zero_first);
        v = xin[j];
    }
    xout[p] = v;
}

// Cross-window accumulation in window order (the reference's serial `S .+= ...`, src/lsfft.jl:122,153,187-189),
// one thread per frequency; products are kept unfused so identical channels give coherence == 1 exactly (Q8/H7).
__global__ void k_window_accum(int kind, const double* __restrict__ X, long long strideB, int Np, int nwin, int Nf,
                               int zero_first, double* __restrict__ sums) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= Nf) return;
    int pc = (k >> 6) * 128 + (k & 63);
    bool noim = zero_first && k == 0;
    if (kind == LPVS_WIN_PSD) {
        double s = sums[k];
        for (int wdx = 0; wdx < nwin; wdx++) {
            const double* x = X + (long long)wdx * strideB;
            double re = x[pc], im = noim ? 0.0 : x[pc + 64];
            s = __dadd_rn(s, __dadd_rn(__dmul_rn(re, re), __dmul_rn(im, im)));
        }
        sums[k] = s;
    } else if (kind == LPVS_WIN_CSD) {
        double sr = sums[k], si = sums[Nf + k];
        for (int wdx = 0; wdx < nwin; wdx++) {
            const double* x = X + (long long)wdx * strideB;
            double ar = x[pc], ai = noim ? 0.0 : x[pc + 64];
            double br = x[Np + pc], bi = noim ? 0.0 : x[Np + pc + 64];
            sr = __dadd_rn(sr, __dadd_rn(__dmul_rn(ar, br), __dmul_rn(ai, bi)));
            si = __dadd_rn(si, __dsub_rn(__dmul_rn(ai, br), __dmul_rn(ar, bi)));
        }
        sums[k] = sr;
        sums[Nf + k] = si;
    } else {
        double syy = sums[k], suu = sums[Nf + k], sr = sums[2 * Nf + k], si = sums[3 * Nf + k];
        for (int wdx = 0; wdx < nwin; wdx++) {
            const double* x = X + (long long)wdx * strideB;
            double ar = x[pc], ai = noim ? 0.0 : x[pc + 64];
            double br = x[Np + pc], bi = noim ? 0.0 : x[Np + pc + 64];
            sr = __dadd_rn(sr, __dadd_rn(__dmul_rn(ar, br), __dmul_rn(ai, bi)));
            si = __dadd_rn(si, __dsub_rn(__dmul_rn(ai, br), __dmul_rn(ar, bi)));
            syy = __dadd_rn(syy, __dadd_rn(__dmul_rn(ar, ar), __dmul_rn(ai, ai)));
            suu = __dadd_rn(suu, __dadd_rn(__dmul_rn(br, br), __dmul_rn(bi, bi)));
        }
        sums[k] = syy;
        sums[Nf + k] = suu;
        sums[2 * Nf + k] = sr;
        sums[3 * Nf + k] = si;
    }
}

// The C x C cross-spectral matrix per frequency: sums[f][i][j] += x_i conj(x_j) over the batch's windows in window order,
// continuing from the previous batch, with k_window_accum's unfused arithmetic (X: [window][channel][Np]).  One thread per
// (f, i <= j); (j, i) is written as the conjugate, so S is exactly Hermitian and S_ii has an exactly zero imaginary part.
__global__ void k_window_matrix_accum(const double* __restrict__ X, long long strideB, int Np, int C, int nwin, int Nf,
                                      int zero_first, double* __restrict__ sums) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)Nf * C * C) return;
    const int k = (int)(idx / ((long long)C * C)), i = (int)(idx / C % C), j = (int)(idx % C);
    if (i > j) return;
    const int pc = (k >> 6) * 128 + (k & 63);
    const bool noim = zero_first && k == 0;
    double* sij = sums + 2 * (((long long)k * C + i) * C + j);
    double sr = sij[0], si = sij[1];
    for (int wdx = 0; wdx < nwin; wdx++) {
        const double* xi = X + (long long)wdx * strideB + (long long)i * Np;
        const double* xj = X + (long long)wdx * strideB + (long long)j * Np;
        const double ar = xi[pc], ai = noim ? 0.0 : xi[pc + 64];
        const double br = xj[pc], bi = noim ? 0.0 : xj[pc + 64];
        sr = __dadd_rn(sr, __dadd_rn(__dmul_rn(ar, br), __dmul_rn(ai, bi)));
        si = __dadd_rn(si, __dsub_rn(__dmul_rn(ai, br), __dmul_rn(ar, bi)));
    }
    sij[0] = sr;
    sij[1] = si;
    if (i != j) {
        double* sji = sums + 2 * (((long long)k * C + j) * C + i);
        sji[0] = sr;
        sji[1] = -si;
    }
}

// ---------------------------------------------------------------------------------------------------------
// single-problem Gram (with sample splitting) and factor/solve
// ---------------------------------------------------------------------------------------------------------
void fill_basis_args(const FourierPlan& pl, GramArgs& g) {
    g.ncc = pl.Nf;
    g.nblk = pl.nblk;
    g.f = pl.d_f;
    g.wtab = pl.d_wtab;
    g.gscale = pl.dd * pl.dd;
    g.bscale = pl.dd;
    g.E = nullptr;
    g.Kt = nullptr;
    g.lpv_nf = 1;
}

// LPVS_PHASE_STRUCTURED: the sums of `nprob` problems described by g (samples, weights, right-hand sides, problem ranges) into Z
static int structured_sums(lpvs_ctx* c, const FourierPlan& pl, const StructuredLayout& lay, const GramArgs& g, int nprob,
                           double2* Z) {
    double2* tab = ws<double2>(c, BUF_SANC, (size_t)lay.nrows * g.tbl_ns);
    if (!tab) return fail(c, LPVS_E_NOMEM, "out of device memory (sum tables)");
    launch_sum_tables(g.t, g.tbl_base, g.tbl_ns, pl.d_sfreq, lay.nzb, structured_layout(pl.f0, pl.Nf, 2).nzb, tab, c->st);
    SumArgs a{};
    a.t = g.t;
    a.W = g.W;
    a.y = g.y;
    a.u = g.u;
    a.w_abs = g.w_abs;
    a.start0 = g.start0;
    a.hop = g.hop;
    a.n = g.n;
    a.s_end = g.s_end;
    a.tab = tab;
    a.tbl_base = g.tbl_base;
    a.tbl_ns = g.tbl_ns;
    a.nzg = lay.nzg;
    a.nby = lay.nby;
    a.nzb = lay.nzb;
    a.Z = Z;
    a.strideZ = (long long)lay.nzb * FB;
    c->launches += 1 + launch_trig_sums(a, nprob, c->st);
    return LPVS_OK;
}
// G (and b when B is given) of `nprob` problems from their sums
static void structured_fill(lpvs_ctx* c, const FourierPlan& pl, const StructuredLayout& lay, const double2* Z, double* G,
                            long long strideG, double* B, long long strideB, int nrhs, int nprob) {
    FillArgs fa{};
    fa.Z = Z;
    fa.strideZ = (long long)lay.nzb * FB;
    fa.zm_off = lay.zm_off;
    fa.zp_off = lay.zp_off;
    fa.zy_off[0] = lay.zy_off[0];
    fa.zy_off[1] = lay.zy_off[1];
    fa.ncc = pl.Nf;
    fa.nblk = pl.nblk;
    fa.zero_first = pl.zero_first;
    fa.gscale = pl.dd * pl.dd;
    fa.G = G;
    fa.strideG = strideG;
    c->launches += launch_gram_fill(fa, nprob, c->st);
    if (B && nrhs > 0) {
        launch_rhs_from_sums(fa, nrhs, pl.dd, B, strideB, nprob, c->st);
        c->launches++;
    }
}

// LPVS_PHASE_STRUCTURED_REF: G += D'B + B'D, b += D'[y u] for the `nprob` problems described by g (corr.cu); G / B as filled
// by structured_fill.  The per-sample tables cover g's table range [g.tbl_base, g.tbl_base + g.tbl_ns); the scales (and with
// them the rounding of the correction) are taken from max |t| over [scal_s0, scal_s0 + scal_ns), the table range if scal_ns = 0.
static int structured_correct(lpvs_ctx* c, const FourierPlan& pl, const GramArgs& g, double* G, long long strideG, double* B,
                              long long strideB, int nrhs, int nprob, long long scal_s0 = 0, long long scal_ns = 0) {
    CorrArgs a{};
    a.t = g.t;
    a.W = g.W;
    a.y = g.y;
    a.u = g.u;
    a.w_abs = g.w_abs;
    a.start0 = g.start0;
    a.hop = g.hop;
    a.n = g.n;
    a.s_end = g.s_end;
    a.ncc = pl.Nf;
    a.nblk = pl.nblk;
    a.nrhs = nrhs;
    a.wtab = pl.d_cwtab;
    a.wmax = pl.cw_max;
    a.dwmax = pl.cdw_max;
    a.df = pl.df;
    a.tbl_base = g.tbl_base;
    a.tbl_ns = g.tbl_ns;
    a.scal_base = scal_s0;
    a.scal_ns = scal_ns;
    const long long ngr = (long long)pl.nblk * (FB / GRP);
    const long long w0 = g.w_abs ? g.tbl_base : 0, nw = g.w_abs ? g.tbl_ns : g.n;
    a.scal = ws<double>(c, BUF_CSCAL, 2);
    a.eps = ws<uint4>(c, BUF_CEPS, (size_t)ngr * g.tbl_ns);
    a.anc = ws<float2>(c, BUF_CANC, (size_t)ngr * g.tbl_ns);
    a.step = ws<float2>(c, BUF_CSTEP, (size_t)g.tbl_ns);
    a.wf = ws<float>(c, BUF_CWF, (size_t)nw);
    if (!a.scal || !a.eps || !a.anc || !a.step || !a.wf) return fail(c, LPVS_E_NOMEM, "out of device memory (correction tables)");
    a.gscale = pl.dd * pl.dd;
    a.bscale = pl.dd;
    a.G = G;
    a.strideG = strideG;
    a.B = B;
    a.strideB = strideB;
    c->launches += launch_corr_tables(a, w0, nw, c->st);
    c->launches += launch_gram_corr(a, nprob, c->st);
    if (B && nrhs > 0 && g.y) c->launches += launch_rhs_corr(a, nprob, c->st);
    LPVS_CU(c, cudaGetLastError());
    return LPVS_OK;
}

// gram_single for LPVS_PHASE_STRUCTURED: the sums are additive over sample splits (and over table segments); G and b are
// filled once from the totals
static int gram_single_structured(lpvs_ctx* c, const FourierPlan& pl, const double* d_t, const double* d_y,
                                  const double* d_u, const double* d_W, int64_t N, int nrhs, double* d_G, double* d_B) {
    if (!d_B || !d_y) nrhs = 0;
    if (nrhs > 1 && !d_u) nrhs = 1;
    const StructuredLayout lay = structured_layout(pl.f0, pl.Nf, nrhs);
    const long long nz64 = (long long)lay.nzb * FB;
    const long long per_sample = (long long)lay.nrows * sizeof(double2);
    const long long seg_cap = std::max<long long>(65536, (8LL << 30) / per_sample);
    const int nseg = (int)std::max<long long>(1, (N + seg_cap - 1) / seg_cap);
    const long long seg_len = (N + nseg - 1) / nseg;
    // enough CTAs (nzb per split) to fill the machine a few times over, each split >= 2048 samples
    const long long want = (8LL * c->sms + lay.nzb - 1) / lay.nzb, maxs = std::max<long long>(1, seg_len / 2048);
    const int nsplit = (int)std::min(want, maxs);
    double2* Zacc = ws<double2>(c, BUF_ZSUM, (size_t)nz64);
    double2* Zparts = ws<double2>(c, BUF_ZPART, (size_t)nsplit * nz64);
    if (!Zacc || !Zparts) return fail(c, LPVS_E_NOMEM, "out of device memory (structured Gram)");
    gram_timer_begin(c);
    for (int sgi = 0; sgi < nseg; sgi++) {
        const long long s0 = sgi * seg_len, s1 = std::min<long long>(N, s0 + seg_len);
        if (s1 <= s0) break;
        const long long ns = s1 - s0;
        long long n_split = (ns + nsplit - 1) / nsplit;
        n_split = (n_split + KC - 1) / KC * KC;
        const int nprob = (int)((ns + n_split - 1) / n_split);
        GramArgs g{};
        g.t = d_t;
        g.y = d_y;
        g.u = d_u;
        g.W = d_W;
        g.w_abs = 1;
        g.start0 = s0;
        g.hop = n_split;
        g.n = (int)n_split;
        g.s_end = s1;
        g.tbl_base = s0;
        g.tbl_ns = ns;
        int rc = structured_sums(c, pl, lay, g, nprob, Zparts);
        if (rc) return rc;
        launch_sum_parts(Zacc, Zparts, (int)nz64, nz64, nprob, sgi > 0, c->st);
        c->launches++;
    }
    structured_fill(c, pl, lay, Zacc, d_G, 0, d_B, 0, nrhs, 1);
    if (pl.structured_ref) {
        // Sample splits into zeroed partial buffers (each CTA read-modify-writes its own tile), added in split order.  The
        // per-sample tables are built segment by segment (<= 4 GiB); every segment accumulates into the same partials.
        const long long Np = pl.Np, part_stride = Np * Np + 2 * Np;
        const int ntiles = pl.nblk * (pl.nblk + 1) / 2;
        const long long per_s = (long long)corr_table_bytes_per_sample(pl.nblk) + 4;
        const long long cseg_cap = std::max<long long>(65536, (4LL << 30) / per_s);
        const int ncseg = (int)std::max<long long>(1, (N + cseg_cap - 1) / cseg_cap);
        const long long cseg_len = (N + ncseg - 1) / ncseg;
        const long long wantc = (4LL * c->sms + ntiles - 1) / ntiles, maxc = std::max<long long>(1, cseg_len / 2048);
        const int ncs = (int)std::min(wantc, maxc);
        long long n_split = (cseg_len + ncs - 1) / ncs;
        n_split = (n_split + KC - 1) / KC * KC;
        const int nprob_max = (int)((cseg_len + n_split - 1) / n_split);
        const bool direct = ncseg == 1 && nprob_max == 1;
        double* parts = nullptr;
        if (!direct) {
            parts = ws<double>(c, BUF_CPART, (size_t)nprob_max * part_stride);
            if (!parts) return fail(c, LPVS_E_NOMEM, "out of device memory (correction partials)");
            LPVS_CU(c, cudaMemsetAsync(parts, 0, sizeof(double) * nprob_max * part_stride, c->st));
        }
        for (int sgi = 0; sgi < ncseg; sgi++) {
            const long long s0 = sgi * cseg_len, s1 = std::min<long long>(N, s0 + cseg_len);
            if (s1 <= s0) break;
            GramArgs g{};
            g.t = d_t;
            g.y = nrhs > 0 ? d_y : nullptr;
            g.u = nrhs > 1 ? d_u : nullptr;
            g.W = d_W;
            g.w_abs = 1;
            g.start0 = s0;
            g.hop = n_split;
            g.n = (int)n_split;
            g.s_end = s1;
            g.tbl_base = s0;
            g.tbl_ns = s1 - s0;
            const int nprob = (int)((s1 - s0 + n_split - 1) / n_split);
            int rc = direct ? structured_correct(c, pl, g, d_G, 0, d_B, 0, nrhs, 1)
                            : structured_correct(c, pl, g, parts, part_stride, parts + Np * Np, part_stride, nrhs, nprob);
            if (rc) return rc;
        }
        if (!direct) {
            reduce_parts(c, d_G, parts, Np * Np, part_stride, nprob_max, 1);
            if (d_B && nrhs > 0) reduce_parts(c, d_B, parts + Np * Np, 2 * Np, part_stride, nprob_max, 1);
        }
    }
    gram_timer_end(c, (double)N * nz64 * 8.0, 1);  // executed: one complex rotation + accumulation per (sample, sum)
    LPVS_CU(c, cudaGetLastError());
    return LPVS_OK;
}

// the chain anchor tables of g.t over g's table range [g.tbl_base, g.tbl_base + g.tbl_ns), into g.anc / g.del
static int anchor_tables(lpvs_ctx* c, const FourierPlan& pl, GramArgs& g) {
    double2* anc = ws<double2>(c, BUF_ANC, (size_t)pl.ngroups * g.tbl_ns);
    double2* del = ws<double2>(c, BUF_DEL, (size_t)g.tbl_ns);
    if (!anc || !del) return fail(c, LPVS_E_NOMEM, "out of device memory (anchor table)");
    launch_anchor_table(g.t, g.tbl_base, g.tbl_ns, pl.d_f, pl.nblk, pl.df, anc, del, c->st);
    c->launches++;
    g.anc = anc;
    g.del = del;
    return LPVS_OK;
}

int gram_single(lpvs_ctx* c, const FourierPlan& pl, const double* d_t, const double* d_y, const double* d_u,
                const double* d_W, int64_t N, int nrhs, double* d_G, double* d_B) {
    if (pl.structured) return gram_single_structured(c, pl, d_t, d_y, d_u, d_W, N, nrhs, d_G, d_B);
    const long long Np = pl.Np;
    const int ntiles = pl.nblk * (pl.nblk + 1) / 2;
    // split over samples when tiles alone cannot fill the machine; each split >= 2048 samples.  Among the admissible split
    // counts take the one whose CTA count wastes the least of its last wave (36 tiles x 17 splits = 4.14 waves ran cfg5b's
    // Gram at 76 % of peak; x 37 = exactly 9 waves)
    auto pick_split = [&](long long nsamp) {
        if (ntiles >= 4 * c->sms) return 1;
        const long long want = (4LL * c->sms + ntiles - 1) / ntiles;
        const long long maxs = std::max<long long>(1, nsamp / 2048);
        if (maxs <= want) return (int)maxs;
        int best = (int)want;
        double best_eff = 0.0;
        for (long long sct = want; sct <= std::min(maxs, 3 * want); sct++) {
            const long long ctas = sct * ntiles, waves = (ctas + c->sms - 1) / c->sms;
            const double eff = (double)ctas / (double)(waves * c->sms);
            if (eff > best_eff + 1e-9) {
                best_eff = eff;
                best = (int)sct;
            }
        }
        return best;
    };
    const int nsplit = pick_split(N);
    // segment the sample axis so the anchor table stays below ~16 GiB (of 180 GB HBM)
    long long seg_cap = N;
    if (gram_is_chain(pl.mode)) {
        long long per_sample = (long long)(pl.ngroups + 1) * sizeof(double2);
        seg_cap = std::max<long long>(65536, (16LL << 30) / per_sample);
    }
    int nseg = (int)((N + seg_cap - 1) / seg_cap);
    if (nseg < 1) nseg = 1;
    long long seg_len = (N + nseg - 1) / nseg;
    // segments run one after the other, so EACH must be split enough to fill the machine on its own
    const int split_per_seg = nseg == 1 ? nsplit : pick_split(seg_len);
    const bool direct_out = (nseg == 1 && split_per_seg == 1);
    double* parts = nullptr;
    const long long part_stride = Np * Np + 2 * Np;
    if (!direct_out) {
        parts = ws<double>(c, BUF_PART, (size_t)split_per_seg * part_stride);
        if (!parts) return fail(c, LPVS_E_NOMEM, "out of device memory (Gram partials)");
    }
    for (int sgi = 0; sgi < nseg; sgi++) {
        long long s0 = sgi * seg_len, s1 = std::min<long long>(N, s0 + seg_len);
        if (s1 <= s0) break;
        long long ns = s1 - s0;
        long long n_split = (ns + split_per_seg - 1) / split_per_seg;
        n_split = (n_split + KC - 1) / KC * KC;
        int nprob = (int)((ns + n_split - 1) / n_split);
        GramArgs g{};
        fill_basis_args(pl, g);
        g.t = d_t;
        g.y = d_y;
        g.u = d_u;
        g.W = d_W;
        g.w_abs = 1;
        g.start0 = s0;
        g.hop = n_split;
        g.n = (int)n_split;
        g.s_end = s1;
        g.nrhs = nrhs;
        g.tbl_base = s0;
        g.tbl_ns = ns;
        int rc;
        if (gram_is_chain(pl.mode) && (rc = anchor_tables(c, pl, g))) return rc;
        if (direct_out) {
            g.G = d_G;
            g.strideG = 0;
            g.B = d_B;
            g.strideB = 0;
        } else {
            g.G = parts;
            g.strideG = part_stride;
            g.B = parts + Np * Np;
            g.strideB = part_stride;
        }
        gram_timer_begin(c);
        c->launches += launch_gram(pl.mode, g, nprob, c->st);
        gram_timer_end(c, (double)ns * pl.Nreg * (pl.Nreg + 1.0), 1);
        if (!direct_out) {
            k_reduce_parts<<<(unsigned)((Np * Np + 255) / 256), 256, 0, c->st>>>(d_G, parts, Np * Np, part_stride,
                                                                                 nprob, sgi > 0);
            if (d_B)
                k_reduce_parts<<<(unsigned)((2 * Np + 255) / 256), 256, 0, c->st>>>(d_B, parts + Np * Np, 2 * Np,
                                                                                    part_stride, nprob, sgi > 0);
            c->launches += 2;
        }
    }
    LPVS_CU(c, cudaGetLastError());
    return LPVS_OK;
}

int factor_solve(lpvs_ctx* c, int ncc, int zero_first, int Np, double* d_G, double* d_B, int nrhs, double ridge,
                 int nproblems, int* info_host, const double* d_maxdiag, double tol_scale, const double* d_ridge,
                 bool robust) {
    const int nb = Np / TB;
    CholArgs ca{};
    ca.G = d_G;
    ca.strideG = (long long)Np * Np;
    ca.Y = nullptr;
    ca.strideY = 0;
    ca.Linv = ws<double>(c, BUF_LINV, (size_t)nproblems * nb * TB * TB);
    ca.strideLinv = (long long)nb * TB * TB;
    ca.info = ws<int>(c, BUF_INFO, (size_t)nproblems);
    ca.Np = Np;
    ca.nb = nb;
    ca.maxdiag = d_maxdiag;
    ca.tol_scale = tol_scale;
    robust = robust && nproblems == 1;
    if (robust) {
        ca.trsm_scratch = ws<double>(c, BUF_TRSM, (size_t)nb * TB * TB);
        if (!ca.trsm_scratch) return fail(c, LPVS_E_NOMEM, "out of device memory (TRSM refinement scratch)");
    }
    const bool fuse_fwd = d_B && nrhs > 0 && !robust;  // L y = b rides along with the factorisation
    if (fuse_fwd) {
        ca.rhs = d_B;
        ca.strideRhs = 2LL * Np;
        ca.nrhs = nrhs;
    }
    if (!ca.Linv || !ca.info) return fail(c, LPVS_E_NOMEM, "out of device memory (factor workspace)");
    LPVS_CU(c, cudaMemsetAsync(ca.info, 0, sizeof(int) * nproblems, c->st));
    launch_diag_prepare(d_G, ca.strideG, Np, ncc, zero_first, d_ridge, ridge, nproblems, c->st);
    c->launches += 1 + potrf(ca, nproblems, c->sms, c->st, &c->la);
    if (d_B && nrhs > 0) {
        launch_trsv(ca, d_B, 2LL * Np, nrhs, nproblems, c->st, fuse_fwd,
                    nproblems == 1 ? trsv_flags(c, nb) : nullptr);
        c->launches++;
    }
    LPVS_CU(c, cudaGetLastError());
    if (info_host)
        LPVS_CU(c, cudaMemcpyAsync(info_host, ca.info, sizeof(int) * nproblems, cudaMemcpyDeviceToHost, c->st));
    return LPVS_OK;
}

// flags a NaN / Inf in the n uploaded doubles at d (device) for inputs_finite
static void scan_finite(lpvs_ctx* c, const double* d, long long n) {
    if (!c->d_nonfinite || n <= 0) return;
    k_check_finite<<<(int)std::min<long long>((n + 255) / 256, 1184), 256, 0, c->st>>>(d, n, c->d_nonfinite);
    c->launches++;
}

int upload(lpvs_ctx* c, int slot, const double* h, int64_t n, double** d) {
    *d = nullptr;
    if (!h) return LPVS_OK;
    double* p = ws<double>(c, slot, (size_t)n);
    if (!p) return fail(c, LPVS_E_NOMEM, "out of device memory (input upload, %lld doubles)", (long long)n);
    LPVS_CU(c, cudaMemcpyAsync(p, h, sizeof(double) * n, cudaMemcpyHostToDevice, c->st));
    scan_finite(c, p, n);
    *d = p;
    return LPVS_OK;
}

// samples [s0, s0 + ns) of C host channels (channel c at Y + c ldY) to the device, channel c at *d_Y + c ns.  One copy per
// channel: a 2D copy's source pitch (ldY * 8 bytes) is capped near 2 GiB, the ABI's ldY is not.
static int upload_channels(lpvs_ctx* c, const double* Y, int C, int64_t ldY, int64_t s0, int64_t ns, double** d_Y) {
    double* p = ws<double>(c, BUF_Y, (size_t)C * ns);
    if (!p) return fail(c, LPVS_E_NOMEM, "out of device memory (input upload, %d x %lld doubles)", C, (long long)ns);
    for (int ch = 0; ch < C; ch++)
        LPVS_CU(c, cudaMemcpyAsync(p + (size_t)ch * ns, Y + (size_t)ch * ldY + s0, sizeof(double) * ns,
                                   cudaMemcpyHostToDevice, c->st));
    *d_Y = p;
    return LPVS_OK;
}

int inputs_finite(lpvs_ctx* c) {
    int h = 0;
    if (c->d_nonfinite) LPVS_CU(c, cudaMemcpyAsync(&h, c->d_nonfinite, sizeof(int), cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    if (h & 2)
        return fail(c, LPVS_E_NONFINITE,
                    "LPV basis normalisation is 0/0 for some sample: with coulomb=true a scheduling value whose sign "
                    "matches no centre (V == 0) activates no basis function (the reference returns NaNs here)");
    if (h) return fail(c, LPVS_E_NONFINITE, "non-finite value (NaN/Inf) in an input array");
    return LPVS_OK;
}

}  // namespace lpvs

using namespace lpvs;

extern "C" {

int lpvs_version(void) { return 100; }

int lpvs_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int lpvs_init(int device, lpvs_ctx** out) {
    if (!out) return LPVS_E_BAD_ARG;
    *out = nullptr;
    int n = lpvs_device_count();
    if (n <= 0 || device < 0 || device >= n) return LPVS_E_CUDA;  // no CPU fallback
    if (cudaSetDevice(device) != cudaSuccess) return LPVS_E_CUDA;
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, device) != cudaSuccess) return LPVS_E_CUDA;
    if (p.major < 10) return LPVS_E_UNSUPPORTED;  // sm_100a only
    lpvs_ctx* c = new lpvs_ctx();
    c->device = device;
    c->sms = p.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->own_st, cudaStreamNonBlocking) != cudaSuccess) {
        delete c;
        return LPVS_E_CUDA;
    }
    c->st = c->own_st;
    cudaStreamCreateWithFlags(&c->la.aux, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&c->la.e_trsm, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->la.e_rest, cudaEventDisableTiming);
    cudaEventCreate(&c->ev_call0);
    cudaEventCreate(&c->ev_call1);
    if (cudaMalloc(&c->d_nonfinite, sizeof(int)) != cudaSuccess) c->d_nonfinite = nullptr;
    *out = c;
    return LPVS_OK;
}

void lpvs_destroy(lpvs_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    admm_release_all(c);
    cudaStreamSynchronize(c->st);
    for (auto& b : c->buf)
        if (b.p) cudaFree(b.p);
    for (auto e : c->ev) cudaEventDestroy(e);
    cudaFree(c->d_nonfinite);
    cudaEventDestroy(c->ev_call0);
    cudaEventDestroy(c->ev_call1);
    cudaStreamDestroy(c->own_st);
    if (c->la.aux) cudaStreamDestroy(c->la.aux);
    if (c->la.e_trsm) cudaEventDestroy(c->la.e_trsm);
    if (c->la.e_rest) cudaEventDestroy(c->la.e_rest);
    delete c;
}

const char* lpvs_last_error(const lpvs_ctx* c) { return c ? c->err.c_str() : "no context (no CUDA device?)"; }

int lpvs_set_option(lpvs_ctx* c, int key, double value) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    switch (key) {
        case LPVS_OPT_PHASE_MODE:
            if ((int)value < LPVS_PHASE_AUTO || (int)value > LPVS_PHASE_STRUCTURED_REF)
                return fail(c, LPVS_E_BAD_ARG, "LPVS_OPT_PHASE_MODE must be one of lpvs_phase_mode (0 .. %d)", (int)LPVS_PHASE_STRUCTURED_REF);
            c->phase_mode = (int)value;
            break;
        case LPVS_OPT_WINDOW_BATCH: c->window_batch = (int)value; break;
        case LPVS_OPT_JITTER: c->jitter = (int)value; break;
        case LPVS_OPT_ADMM_CHECK_EVERY: c->admm_check_every = std::max(1, (int)value); break;
        case LPVS_OPT_ADMM_SYMV: c->admm_symv = (int)value; break;
        case LPVS_OPT_TRSV_FLOW: c->trsv_flow = (int)value != 0; break;
        case LPVS_OPT_ADMM_M32: c->admm_m32 = (int)value != 0; break;
        case LPVS_OPT_SHARD_EXCHANGE:
            if ((int)value < 0 || (int)value > 2) return fail(c, LPVS_E_BAD_ARG, "LPVS_OPT_SHARD_EXCHANGE must be 0, 1 or 2");
            c->shard_exchange = (int)value;
            break;
        default: return fail(c, LPVS_E_BAD_ARG, "unknown option %d", key);
    }
    return LPVS_OK;
}

int lpvs_set_stream(lpvs_ctx* c, void* stream) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->st);
    c->st = stream ? (cudaStream_t)stream : c->own_st;
    return LPVS_OK;
}

int64_t lpvs_launch_count(const lpvs_ctx* c) { return c ? c->launches : 0; }

int lpvs_last_gram_timing(const lpvs_ctx* c, double* ms, int64_t* launches, double* flops) {
    if (!c) return LPVS_E_BAD_ARG;
    if (ms) *ms = c->gram_ms;
    if (launches) *launches = c->gram_launches;
    if (flops) *flops = c->gram_flops;
    return LPVS_OK;
}

int lpvs_last_call_ms(const lpvs_ctx* c, double* ms) {
    if (!c || !ms) return LPVS_E_BAD_ARG;
    float m = 0.f;
    if (cudaEventSynchronize(c->ev_call1) != cudaSuccess || cudaEventElapsedTime(&m, c->ev_call0, c->ev_call1) != cudaSuccess) {
        cudaGetLastError();
        return LPVS_E_CUDA;
    }
    *ms = m;
    return LPVS_OK;
}

int lpvs_dev_alloc(lpvs_ctx* c, int64_t bytes, void** dptr) {
    if (!c || !dptr) return LPVS_E_BAD_ARG;
    cudaSetDevice(c->device);
    LPVS_CU(c, cudaMalloc(dptr, (size_t)bytes));
    return LPVS_OK;
}
int lpvs_dev_free(lpvs_ctx* c, void* dptr) {
    if (!c) return LPVS_E_BAD_ARG;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->st);
    LPVS_CU(c, cudaFree(dptr));
    return LPVS_OK;
}
int lpvs_dev_upload(lpvs_ctx* c, void* dptr, const void* hptr, int64_t bytes) {
    if (!c) return LPVS_E_BAD_ARG;
    cudaSetDevice(c->device);
    LPVS_CU(c, cudaMemcpyAsync(dptr, hptr, (size_t)bytes, cudaMemcpyHostToDevice, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    return LPVS_OK;
}
int lpvs_dev_download(lpvs_ctx* c, void* hptr, const void* dptr, int64_t bytes) {
    if (!c) return LPVS_E_BAD_ARG;
    cudaSetDevice(c->device);
    LPVS_CU(c, cudaMemcpyAsync(hptr, dptr, (size_t)bytes, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    return LPVS_OK;
}
int lpvs_release_workspace(lpvs_ctx* c) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    cudaSetDevice(c->device);
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    for (auto& b : c->buf) {
        if (b.p) cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    return LPVS_OK;
}
int lpvs_sync(lpvs_ctx* c) {
    if (!c) return LPVS_E_BAD_ARG;
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    return LPVS_OK;
}

int64_t lpvs_window_count(int64_t N, int n, int noverlap) {
    if (n <= 0) return 0;
    if (noverlap < 0) noverlap = n >> 1;
    if (noverlap >= n) return -1;
    return N >= n ? (N - n) / (n - noverlap) + 1 : 0;
}

int lpvs_gram_fourier(lpvs_ctx* c, const double* y, const double* t, int64_t N, const double* f, int Nf,
                      const double* W, double* G, double* b) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (!t || N <= 0 || !G) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    gram_timer_reset(c);
    FourierPlan pl;
    int rc = make_fourier_plan(c, f, Nf, &pl);
    if (rc) return rc;
    double *d_t, *d_y, *d_W;
    if ((rc = upload(c, BUF_T, t, N, &d_t))) return rc;
    if ((rc = upload(c, BUF_Y, y, N, &d_y))) return rc;
    if ((rc = upload(c, BUF_W, W, N, &d_W))) return rc;
    const long long Np = pl.Np;
    double* d_G = ws<double>(c, BUF_G, (size_t)Np * Np);
    double* d_B = ws<double>(c, BUF_B, (size_t)2 * Np);
    if (!d_G || !d_B) return fail(c, LPVS_E_NOMEM, "out of device memory (G)");
    if ((rc = gram_single(c, pl, d_t, d_y, nullptr, d_W, N, y ? 1 : 0, d_G, d_B))) return rc;
    double* d_out = ws<double>(c, BUF_MISC, (size_t)pl.Nreg * pl.Nreg + pl.Nreg);
    if (!d_out) return fail(c, LPVS_E_NOMEM, "out of device memory (G out)");
    dim3 grid((pl.Nreg + 127) / 128, pl.Nreg);
    k_gather_ref<<<grid, 128, 0, c->st>>>(d_G, (y && b) ? d_B : nullptr, pl.Np, pl.Nf, pl.zero_first, pl.Nreg, d_out,
                                          (y && b) ? d_out + (size_t)pl.Nreg * pl.Nreg : nullptr);
    c->launches++;
    LPVS_CU(c, cudaMemcpyAsync(G, d_out, sizeof(double) * pl.Nreg * pl.Nreg, cudaMemcpyDeviceToHost, c->st));
    if (y && b)
        LPVS_CU(c, cudaMemcpyAsync(b, d_out + (size_t)pl.Nreg * pl.Nreg, sizeof(double) * pl.Nreg,
                                   cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    gram_timer_resolve(c);
    return LPVS_OK;
}

// shared by lpvs_ls_spectral and the ADMM init path: solve one ridge LS on device arrays, x internal in BUF_B
}  // extern "C"

namespace lpvs {
int ls_solve_dev(lpvs_ctx* c, const FourierPlan& pl, const double* d_t, const double* d_y, const double* d_u,
                        const double* d_W, int64_t N, int nrhs, double ridge, bool allow_jitter, double** d_x,
                        int* info) {
    const long long Np = pl.Np;
    double* d_G = ws<double>(c, BUF_G, (size_t)Np * Np);
    double* d_B = ws<double>(c, BUF_B, (size_t)2 * Np);
    double* d_md = ws<double>(c, BUF_SUMS, 8);
    if (!d_G || !d_B || !d_md) return fail(c, LPVS_E_NOMEM, "out of device memory (G)");
    int rc;
    if (info) *info = 0;
    if (!d_W && nrhs == 1 && allow_jitter) {
        // unweighted: the reference solves on [A; lam I] itself (SVD, src/utilities.jl:58) -> operator-accurate solve
        auto regram = [&]() { return gram_single(c, pl, d_t, d_y, nullptr, nullptr, N, 1, d_G, d_B); };
        if ((rc = regram())) return rc;
        OpArgs op;
        op.mode = GRAM_DIRECT;
        op.t = d_t;
        op.f = pl.d_f;
        op.dd = pl.dd;
        op.ncc = pl.Nf;
        op.zero_first = pl.zero_first;
        op.N = N;
        if ((rc = ls_solve_accurate(c, op, pl.Np, pl.zero_first, d_y, d_G, d_B, sqrt(ridge), regram, info))) return rc;
        *d_x = d_B;
        return LPVS_OK;
    }
    double* d_keep = nullptr;  // pristine copy of G, b for the jitter retry (no second Gram pass)
    for (int attempt = 0; attempt < 2; attempt++) {
        if (attempt == 0) {
            if ((rc = gram_single(c, pl, d_t, d_y, d_u, d_W, N, nrhs, d_G, d_B))) return rc;
            if (allow_jitter) {
                d_keep = ws<double>(c, BUF_YINV, (size_t)Np * Np + 2 * Np);
                if (d_keep) {
                    LPVS_CU(c, cudaMemcpyAsync(d_keep, d_G, sizeof(double) * Np * Np, cudaMemcpyDeviceToDevice, c->st));
                    LPVS_CU(c, cudaMemcpyAsync(d_keep + Np * Np, d_B, sizeof(double) * 2 * Np, cudaMemcpyDeviceToDevice,
                                               c->st));
                }
            }
        } else if (d_keep) {
            LPVS_CU(c, cudaMemcpyAsync(d_G, d_keep, sizeof(double) * Np * Np, cudaMemcpyDeviceToDevice, c->st));
            LPVS_CU(c, cudaMemcpyAsync(d_B, d_keep + Np * Np, sizeof(double) * 2 * Np, cudaMemcpyDeviceToDevice, c->st));
        } else {
            if ((rc = gram_single(c, pl, d_t, d_y, d_u, d_W, N, nrhs, d_G, d_B))) return rc;
        }
        double maxdiag = 0.0;
        if (attempt == 0 && allow_jitter) {
            launch_max_diag(d_G, Np * Np, pl.Np, pl.Nf, pl.zero_first, d_md, 1, c->st);
            c->launches++;
        }
        int pinfo = 0;
        // with the jitter policy on, the first attempt also rejects numerically-zero pivots
        // (<= Nreg*eps*max diag G): a tiny positive pivot would otherwise let null-space garbage through
        const bool ranktest = attempt == 0 && allow_jitter;
        if ((rc = factor_solve(c, pl.Nf, pl.zero_first, pl.Np, d_G, d_B, nrhs, ridge, 1, &pinfo,
                               ranktest ? d_md : nullptr, (double)pl.Nreg * 2.220446049250313e-16)))
            return rc;
        if (attempt == 0 && allow_jitter)
            LPVS_CU(c, cudaMemcpyAsync(&maxdiag, d_md, sizeof(double), cudaMemcpyDeviceToHost, c->st));
        LPVS_CU(c, cudaStreamSynchronize(c->st));
        if (pinfo == 0) break;
        if (attempt == 0 && allow_jitter) {
            // SURVEY H1: numerically rank-deficient Gram -> re-factor on device with a jitter ridge
            double jr = (double)pl.Nreg * 2.220446049250313e-16 * maxdiag;
            ridge = std::max(ridge, jr);
            if (info) *info = LPVS_INFO_JITTER;
            continue;
        }
        if (info) *info = pinfo;
        return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown at internal pivot %d (A'WA + ridge not positive definite)",
                    pinfo);
    }
    *d_x = d_B;
    return LPVS_OK;
}
void reduce_parts(lpvs_ctx* c, double* out, const double* parts, long long count, long long stride, int nparts,
                  int accumulate) {
    k_reduce_parts<<<(unsigned)((count + 255) / 256), 256, 0, c->st>>>(out, parts, count, stride, nparts, accumulate);
    c->launches++;
}
void launch_gather_ref(lpvs_ctx* c, const double* G, const double* B, int Np, int half, int zero_first, int nref,
                       double* Gout, double* bout) {
    dim3 grid((nref + 127) / 128, nref);
    k_gather_ref<<<grid, 128, 0, c->st>>>(G, B, Np, half, zero_first, nref, Gout, bout);
    c->launches++;
}
void launch_x_to_complex(lpvs_ctx* c, const double* X, int Np, int ncx, int zero_first, int nrhs, double* out) {
    k_x_to_complex<<<(ncx + 127) / 128, 128, 0, c->st>>>(X, Np, ncx, zero_first, nrhs, out);
    c->launches++;
}
void launch_scatter_ref_vec(lpvs_ctx* c, const double* xin, int half, int zero_first, int nref, int Np, double* xout) {
    k_scatter_ref_vec<<<(Np + 255) / 256, 256, 0, c->st>>>(xin, half, zero_first, nref, Np, xout);
    c->launches++;
}
}  // namespace lpvs

extern "C" {

int lpvs_ls_spectral(lpvs_ctx* c, const double* y, const double* t, int64_t N, const double* f, int Nf,
                     const double* W, double lambda, double* x, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (!y || !t || !x || N <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    gram_timer_reset(c);
    FourierPlan pl;
    int rc = make_fourier_plan(c, f, Nf, &pl);
    if (rc) return rc;
    double *d_t, *d_y, *d_W;
    if ((rc = upload(c, BUF_T, t, N, &d_t))) return rc;
    if ((rc = upload(c, BUF_Y, y, N, &d_y))) return rc;
    if ((rc = upload(c, BUF_W, W, N, &d_W))) return rc;
    // ridge: lambda^2 unweighted (src/utilities.jl:58), lambda weighted (src/lsfft.jl:77)
    double ridge = W ? lambda : lambda * lambda;
    double* d_x;
    // LPVS_OPT_JITTER=1 (default): unweighted -> operator-accurate solve (lsq.cu); weighted -> Cholesky of A'WA + lambda I with
    // a jitter retry on breakdown (the reference's LU at src/lsfft.jl:77 never throws).  0: plain Cholesky, NOT_SPD on breakdown.
    if ((rc = ls_solve_dev(c, pl, d_t, d_y, nullptr, d_W, N, 1, ridge, c->jitter != 0, &d_x, info))) {
        if (inputs_finite(c) == LPVS_E_NONFINITE) return LPVS_E_NONFINITE;  // the more specific diagnosis
        return rc;
    }
    double* d_out = ws<double>(c, BUF_X, (size_t)2 * Nf);
    if (!d_out) return fail(c, LPVS_E_NOMEM, "out of device memory (x)");
    k_x_to_complex<<<(Nf + 127) / 128, 128, 0, c->st>>>(d_x, pl.Np, Nf, pl.zero_first, 1, d_out);
    c->launches++;
    LPVS_CU(c, cudaMemcpyAsync(x, d_out, sizeof(double) * 2 * Nf, cudaMemcpyDeviceToHost, c->st));
    if ((rc = inputs_finite(c))) return rc;
    gram_timer_resolve(c);
    return LPVS_OK;
}

int lpvs_ls_spectral_multi_dev(lpvs_ctx* c, const double* d_Y, int C, int64_t ldY, const double* d_t, int64_t N,
                               const double* f, int Nf, const double* d_W, double lambda, double* X, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (C < 1) return fail(c, LPVS_E_BAD_ARG, "C must be >= 1 (got %d)", C);
    if (!d_Y || !d_t || !X || N <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (ldY < N) return fail(c, LPVS_E_BAD_ARG, "ldY (%lld) must be >= N (%lld)", (long long)ldY, (long long)N);
    std::vector<int> hinfo((size_t)C, 0);
    int* inf = info ? info : hinfo.data();
    for (int ch = 0; ch < C; ch++) inf[ch] = 0;
    gram_timer_reset(c);
    FourierPlan pl;
    int rc = make_fourier_plan(c, f, Nf, &pl);
    if (rc) return rc;
    cudaStream_t st = c->st;
    // non-finite inputs are reported before any work, naming the first channel that holds one
    {
        int* d_flag = ws<int>(c, BUF_MC_ACT, (size_t)std::max(C, 2));
        if (!d_flag) return fail(c, LPVS_E_NOMEM, "out of device memory (flags)");
        int hf[2] = {C, 0};
        LPVS_CU(c, cudaMemcpyAsync(d_flag, hf, sizeof hf, cudaMemcpyHostToDevice, st));
        const unsigned nblk = (unsigned)std::min<long long>((N + 255) / 256, 64);
        k_first_nonfinite_channel<<<dim3(nblk, C), 256, 0, st>>>(d_Y, ldY, N, d_flag);
        k_check_finite<<<nblk, 256, 0, st>>>(d_t, N, d_flag + 1);
        if (d_W) k_check_finite<<<nblk, 256, 0, st>>>(d_W, N, d_flag + 1);
        c->launches += d_W ? 3 : 2;
        LPVS_CU(c, cudaMemcpyAsync(hf, d_flag, sizeof hf, cudaMemcpyDeviceToHost, st));
        LPVS_CU(c, cudaStreamSynchronize(st));
        if (hf[0] < C) return fail(c, LPVS_E_NONFINITE, "non-finite value (NaN/Inf) in channel %d", hf[0]);
        if (hf[1]) return fail(c, LPVS_E_NONFINITE, "non-finite value (NaN/Inf) in t or W");
    }
    const long long Np = pl.Np;
    double* d_G = ws<double>(c, BUF_G, (size_t)Np * Np);
    double* d_Bs = ws<double>(c, BUF_B, (size_t)2 * Np);
    double* d_X = ws<double>(c, BUF_MC_X, (size_t)C * Np);
    if (!d_G || !d_Bs || !d_X) return fail(c, LPVS_E_NOMEM, "out of device memory (G, %d channels)", C);
    // G = A' diag(W) A once for every channel (no right-hand side: those are formed C-wide below)
    auto regram = [&]() { return gram_single(c, pl, d_t, nullptr, nullptr, d_W, N, 0, d_G, d_Bs); };
    if ((rc = regram())) return rc;
    if (!d_W && c->jitter) {
        // unweighted: the operator-accurate solve of lpvs_ls_spectral, its G-only decisions shared (lsq.cu)
        OpArgs op;
        op.mode = GRAM_DIRECT;
        op.t = d_t;
        op.f = pl.d_f;
        op.dd = pl.dd;
        op.ncc = pl.Nf;
        op.zero_first = pl.zero_first;
        op.N = N;
        if ((rc = ls_solve_accurate_multi(c, op, pl.Np, pl.zero_first, d_Y, ldY, C, d_G, lambda, regram, d_X, inf)))
            return rc;
    } else {
        // (A'WA + lambda I) x = A'W y, or (A'A + lambda^2 I) x = A'y with LPVS_OPT_JITTER = 0: one factor, C solves; the
        // jitter retry (a property of G alone) is taken for every channel
        double ridge = d_W ? lambda : lambda * lambda;
        double* d_md = ws<double>(c, BUF_SUMS, 8);
        if (!d_md) return fail(c, LPVS_E_NOMEM, "out of device memory");
        for (int attempt = 0;; attempt++) {
            if (attempt > 0 && (rc = regram())) return rc;
            const bool ranktest = attempt == 0 && c->jitter;
            if (ranktest) {
                launch_max_diag(d_G, Np * Np, pl.Np, pl.Nf, pl.zero_first, d_md, 1, st);
                c->launches++;
            }
            int pinfo = 0;
            double maxdiag = 0.0;
            if ((rc = factor_solve(c, pl.Nf, pl.zero_first, pl.Np, d_G, nullptr, 0, ridge, 1, &pinfo,
                                   ranktest ? d_md : nullptr, (double)pl.Nreg * 2.220446049250313e-16)))
                return rc;
            if (ranktest) LPVS_CU(c, cudaMemcpyAsync(&maxdiag, d_md, sizeof(double), cudaMemcpyDeviceToHost, st));
            LPVS_CU(c, cudaStreamSynchronize(st));
            if (pinfo == 0) break;
            if (ranktest) {
                ridge = std::max(ridge, (double)pl.Nreg * 2.220446049250313e-16 * maxdiag);
                for (int ch = 0; ch < C; ch++) inf[ch] = LPVS_INFO_JITTER;
                continue;
            }
            for (int ch = 0; ch < C; ch++) inf[ch] = pinfo;
            return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown at internal pivot %d (A'WA + ridge not positive definite)",
                        pinfo);
        }
        GramArgs g{};
        fill_basis_args(pl, g);
        g.t = d_t;
        g.W = d_W;
        g.w_abs = 1;
        g.start0 = 0;
        g.s_end = N;
        g.tbl_base = 0;
        g.tbl_ns = N;
        if (gram_is_chain(pl.mode) && (rc = anchor_tables(c, pl, g))) return rc;
        double* d_B = ws<double>(c, BUF_MC_G, (size_t)2 * C * Np);  // B | scratch
        double* d_Li = ws<double>(c, BUF_LSQ_LI, (size_t)Np * Np);
        double* d_S = ws<double>(c, BUF_LSQ_G2, (size_t)Np * Np);
        double* Linv = ws<double>(c, BUF_LINV, (size_t)pl.nblk * TB * TB);
        if (!d_B || !d_Li || !d_S || !Linv) return fail(c, LPVS_E_NOMEM, "out of device memory (solves of %d channels)", C);
        if ((rc = adjoint_apply_multi(c, g, pl.mode, pl.Np, d_Y, ldY, C, d_B))) return rc;
        if ((rc = factor_inverse(c, d_G, Linv, pl.Np, d_Li, d_S))) return rc;
        if ((rc = llt_solve_multi(c, d_Li, pl.Np, d_B, C, nullptr, d_X, d_B + (long long)C * Np))) return rc;
    }
    double* d_out = ws<double>(c, BUF_X, (size_t)2 * Nf * C);
    if (!d_out) return fail(c, LPVS_E_NOMEM, "out of device memory (X)");
    launch_x_to_complex(c, d_X, pl.Np, Nf, pl.zero_first, C, d_out);
    LPVS_CU(c, cudaMemcpyAsync(X, d_out, sizeof(double) * 2 * Nf * C, cudaMemcpyDeviceToHost, st));
    LPVS_CU(c, cudaStreamSynchronize(st));
    gram_timer_resolve(c);
    return LPVS_OK;
}

int lpvs_ls_spectral_multi(lpvs_ctx* c, const double* Y, int C, int64_t ldY, const double* t, int64_t N, const double* f,
                           int Nf, const double* W, double lambda, double* X, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);  // held across upload + compute: the uploaded samples live in the context's workspace
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (C < 1) return fail(c, LPVS_E_BAD_ARG, "C must be >= 1 (got %d)", C);
    if (!Y || !t || !X || N <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (ldY < N) return fail(c, LPVS_E_BAD_ARG, "ldY (%lld) must be >= N (%lld)", (long long)ldY, (long long)N);
    double *d_t, *d_W;
    int rc;
    if ((rc = upload(c, BUF_T, t, N, &d_t))) return rc;
    if ((rc = upload(c, BUF_W, W, N, &d_W))) return rc;
    double* d_Y;
    if ((rc = upload_channels(c, Y, C, ldY, 0, N, &d_Y))) return rc;
    return lpvs_ls_spectral_multi_dev(c, d_Y, C, N, d_t, N, f, Nf, d_W, lambda, X, info);
}

int lpvs_merge_windows(lpvs_ctx* c, const double* pieces, int64_t K, int n, int noverlap, int64_t N, double* out) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (!out || N <= 0 || n <= 0 || K < 0 || (K > 0 && !pieces)) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (noverlap < 0) noverlap = n >> 1;
    if (noverlap >= n) return fail(c, LPVS_E_BAD_ARG, "noverlap must be < n");
    const int hop = n - noverlap;
    if (K > 0 && (K - 1) * (int64_t)hop + n > N) return fail(c, LPVS_E_BAD_ARG, "windows extend beyond the signal");
    double* d_p = nullptr;
    int rc;
    if (K > 0 && (rc = upload(c, BUF_MISC, pieces, K * (int64_t)n, &d_p))) return rc;
    double* d_o = ws<double>(c, BUF_X, (size_t)N);
    if (!d_o) return fail(c, LPVS_E_NOMEM, "out of device memory");
    k_merge_windows<<<(unsigned)((N + 255) / 256), 256, 0, c->st>>>(d_p, K, n, hop, N, d_o);
    c->launches++;
    LPVS_CU(c, cudaMemcpyAsync(out, d_o, sizeof(double) * N, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    return LPVS_OK;
}

int lpvs_tls_spectral(lpvs_ctx* c, const double* y, const double* t, int64_t N, const double* f, int Nf, double* x,
                      int* iters) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (iters) *iters = 0;
    if (!y || !t || !x || N <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    gram_timer_reset(c);
    FourierPlan pl;
    int rc = make_fourier_plan(c, f, Nf, &pl);
    if (rc) return rc;
    double *d_t, *d_y;
    if ((rc = upload(c, BUF_T, t, N, &d_t))) return rc;
    if ((rc = upload(c, BUF_Y, y, N, &d_y))) return rc;
    const long long Np = pl.Np;
    double* d_G = ws<double>(c, BUF_G, (size_t)Np * Np);
    double* d_B = ws<double>(c, BUF_B, (size_t)2 * Np);
    if (!d_G || !d_B) return fail(c, LPVS_E_NOMEM, "out of device memory (G)");
    if ((rc = gram_single(c, pl, d_t, d_y, nullptr, nullptr, N, 1, d_G, d_B))) return rc;
    if ((rc = tls_solve(c, pl.Np, pl.Nf, pl.zero_first, d_y, N, d_G, d_B, iters))) {
        if (inputs_finite(c) == LPVS_E_NONFINITE) return LPVS_E_NONFINITE;
        return rc;
    }
    double* d_out = ws<double>(c, BUF_X, (size_t)2 * Nf);
    if (!d_out) return fail(c, LPVS_E_NOMEM, "out of device memory (x)");
    launch_x_to_complex(c, d_B, pl.Np, Nf, pl.zero_first, 1, d_out);
    LPVS_CU(c, cudaMemcpyAsync(x, d_out, sizeof(double) * 2 * Nf, cudaMemcpyDeviceToHost, c->st));
    if ((rc = inputs_finite(c))) return rc;
    gram_timer_resolve(c);
    return LPVS_OK;
}

static int sums_len(int kind, int Nf) { return kind == LPVS_WIN_PSD ? Nf : (kind == LPVS_WIN_CSD ? 2 * Nf : 4 * Nf); }

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// windowed estimators: the stages of a batch of windows, shared by the dense and sparse, two-channel and matrix paths
// ---------------------------------------------------------------------------------------------------------
namespace lpvs {

// windows [k_begin, k_end) of a record of N samples, n samples each and hop apart: samples [s0, s1)
struct Windows {
    int64_t N;
    int n;
    int64_t hop, k_begin, k_end, s0, s1;
    // the same windows in their own samples [s0, s1), uploaded alone
    Windows uploaded() const { return Windows{s1 - s0, n, hop, 0, k_end - k_begin, 0, s1 - s0}; }
};

// validates the window arguments (noverlap < 0: n / 2, src/windows.jl:29); n > 0 is checked by the caller
static int window_range(lpvs_ctx* c, int64_t N, int n, int noverlap, int64_t k_begin, int64_t k_end, Windows* w) {
    if (noverlap < 0) noverlap = n >> 1;
    if (noverlap >= n) return fail(c, LPVS_E_BAD_ARG, "noverlap must be < n");
    const int64_t K = lpvs_window_count(N, n, noverlap);
    if (k_begin < 0 || k_end > K || k_begin > k_end) return fail(c, LPVS_E_BAD_ARG, "window range out of bounds");
    const int64_t hop = n - noverlap;
    *w = Windows{N, n, hop, k_begin, k_end, k_begin * hop, (k_end - 1) * hop + n};
    return LPVS_OK;
}

// windows per batch: as many as `budget` bytes hold at `per_window` bytes each, with whole_waves rounded down to whole waves
// of the one-CTA-per-window launches (k_potf2, the last TRSM / SYRK steps) so that they fill every SM.  A positive
// LPVS_OPT_WINDOW_BATCH replaces the budget.  At most `cap` and the window count, at least 1.
static int64_t batch_size(lpvs_ctx* c, long long per_window, long long budget, bool whole_waves, int64_t cap,
                          int64_t nwin) {
    int64_t batch = c->window_batch > 0 ? c->window_batch : std::max<int64_t>(1, budget / per_window);
    if (whole_waves && c->window_batch <= 0 && batch > c->sms) batch -= batch % c->sms;
    return std::min<int64_t>(std::min<int64_t>(batch, cap), std::max<int64_t>(1, nwin));
}

// The Gram matrices of windows [k0, k0 + nw) of w into d_G (Np^2 apart) and, when nrhs > 0, their right-hand sides
// A'W [y u] into d_B (2 Np apart), timed by the Gram timer; g is left describing the batch for later passes over it.
// structured_tables: build the chain anchor tables in the structured modes too (k_gram_rhs_multi reads them; without it
// they are built there only for a window re-done alone).  range_scales: LPVS_PHASE_STRUCTURED_REF scales its correction by
// max |t| over all of w's windows, so that a window's bits do not depend on the batch it falls in; else over the batch's.
static int window_gram(lpvs_ctx* c, const FourierPlan& pl, const Windows& w, const double* d_t, const double* d_y,
                       const double* d_u, const double* d_W, int nrhs, int64_t k0, int nw, bool structured_tables,
                       bool range_scales, double* d_G, double* d_B, GramArgs& g) {
    const long long Np = pl.Np, s0 = k0 * w.hop;
    g = GramArgs{};
    fill_basis_args(pl, g);
    g.t = d_t;
    g.y = d_y;
    g.u = nrhs > 1 ? d_u : nullptr;
    g.W = d_W;
    g.w_abs = 0;
    g.start0 = s0;
    g.hop = w.hop;
    g.n = w.n;
    g.s_end = w.N;
    g.nrhs = nrhs;
    g.tbl_base = s0;
    g.tbl_ns = (long long)(nw - 1) * w.hop + w.n;
    g.G = d_G;
    g.strideG = Np * Np;
    g.B = d_B;
    g.strideB = 2 * Np;
    int rc;
    if (gram_is_chain(pl.mode) && (structured_tables || !pl.structured) && (rc = anchor_tables(c, pl, g))) return rc;
    gram_timer_begin(c);
    if (pl.structured) {
        // Gram matrices and right-hand sides from the windows' trigonometric sums (structured.cu)
        const StructuredLayout lay = structured_layout(pl.f0, pl.Nf, nrhs);
        double2* Z = ws<double2>(c, BUF_ZSUM, (size_t)nw * lay.nzb * FB);
        if (!Z) return fail(c, LPVS_E_NOMEM, "out of device memory (window sums)");
        if ((rc = structured_sums(c, pl, lay, g, nw, Z))) return rc;
        structured_fill(c, pl, lay, Z, d_G, Np * Np, d_B, 2 * Np, nrhs, nw);
        if (pl.structured_ref && (rc = structured_correct(c, pl, g, d_G, Np * Np, d_B, 2 * Np, nrhs, nw,
                                                          range_scales ? w.s0 : 0, range_scales ? w.s1 - w.s0 : 0)))
            return rc;
        gram_timer_end(c, (double)nw * w.n * lay.nzb * FB * 8.0, 1);
    } else {
        c->launches += launch_gram(pl.mode, g, nw, c->st);  // k_gram (+ k_gram_rhs when there are two channels)
        gram_timer_end(c, (double)nw * w.n * pl.Nreg * (pl.Nreg + 1.0), 1);
    }
    return LPVS_OK;
}

// The reference's LU of A'WA + lambda I never throws (src/lsfft.jl:77): a numerically singular window i of the batch g
// describes is re-done alone with the jitter ridge max(lambda, Nreg eps max diag G).  Its Gram matrix (and, when
// g.nrhs > 0, its right-hand sides, at *d_g1 + Np^2) is formed again in *d_g1 and factorised there, the right-hand sides
// forward-substituted; the pivot is copied to *pinfo asynchronously.  The caller finishes the solve.
static int jitter_refactor(lpvs_ctx* c, const FourierPlan& pl, GramArgs& g, int i, double lambda, double** d_g1,
                           int* pinfo) {
    const long long Np = pl.Np, nb1 = g.nrhs > 0 ? 2 * Np : 0;
    double* d_g = ws<double>(c, BUF_YINV, (size_t)Np * Np + nb1 + 8);
    if (!d_g) return fail(c, LPVS_E_NOMEM, "out of device memory (window retry)");
    double* d_b = g.nrhs > 0 ? d_g + Np * Np : nullptr;
    double* d_md = d_g + Np * Np + nb1;
    int rc;
    if (gram_is_chain(pl.mode) && !g.anc && (rc = anchor_tables(c, pl, g))) return rc;
    GramArgs g1 = g;
    g1.start0 = g.start0 + (long long)i * g.hop;
    g1.G = d_g;
    g1.B = d_b;
    c->launches += launch_gram(pl.mode, g1, 1, c->st);
    launch_max_diag(d_g, Np * Np, pl.Np, pl.Nf, pl.zero_first, d_md, 1, c->st);
    k_jitter_ridge<<<1, 1, 0, c->st>>>(d_md, lambda, (double)pl.Nreg * 2.220446049250313e-16, d_md + 1);
    c->launches += 2;
    *d_g1 = d_g;
    return factor_solve(c, pl.Nf, pl.zero_first, pl.Np, d_g, d_b, g.nrhs, 0.0, 1, pinfo, nullptr, 0.0, d_md + 1);
}

// M = (A'WA + I/mu)^-1 of the nw windows in d_G, in place (d_Y: the inverse's workspace); the pivots are copied to hinfo
// asynchronously
static int batch_inverse(lpvs_ctx* c, const FourierPlan& pl, double* d_G, double* d_Y, int nw, double mu, int* hinfo) {
    const long long Np = pl.Np;
    const int nb = pl.Np / TB;
    CholArgs ca{};
    ca.G = d_G;
    ca.strideG = Np * Np;
    ca.Y = d_Y;
    ca.strideY = Np * Np;
    ca.Linv = ws<double>(c, BUF_LINV, (size_t)nw * nb * TB * TB);
    ca.strideLinv = (long long)nb * TB * TB;
    ca.info = ws<int>(c, BUF_INFO, (size_t)nw);
    ca.Np = pl.Np;
    ca.nb = nb;
    if (!ca.Linv || !ca.info) return fail(c, LPVS_E_NOMEM, "out of device memory (factor workspace)");
    cudaMemsetAsync(ca.info, 0, sizeof(int) * nw, c->st);
    launch_diag_prepare(d_G, ca.strideG, pl.Np, pl.Nf, pl.zero_first, nullptr, 1.0 / mu, nw, c->st);
    c->launches += 1 + potrf(ca, nw, c->sms, c->st);
    c->launches += potri(ca, nw, c->st);
    cudaMemcpyAsync(hinfo, ca.info, sizeof(int) * nw, cudaMemcpyDeviceToHost, c->st);
    return LPVS_OK;
}

// the first window whose factorisation broke down, by its index in the caller's record, reported as LPVS_E_NOT_SPD
struct FirstFailure {
    int pivot = 0;
    int64_t window = -1;
    void note(int p, int64_t k) {
        if (p && !pivot) {
            pivot = p;
            window = k;
        }
    }
    int report(lpvs_ctx* c, int* info) const {
        if (info) *info = pivot;
        return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown in window %lld at internal pivot %d", (long long)window, pivot);
    }
};

// Declared ahead of a batch loop that copies into host memory (pivots, iteration counts, the caller's residuals): any
// return from the loop then waits for the stream, so that no copy lands after the call has returned.  Cleared once the
// loop has waited for its last copy.
struct HostCopies {
    cudaStream_t st;
    bool pending = true;
    ~HostCopies() {
        if (pending) cudaStreamSynchronize(st);
    }
};

// the samples of w's windows of a host record's t, y and u (nullable) to the device: only this range travels
static int upload_range(lpvs_ctx* c, const Windows& w, const double* t, const double* y, const double* u, double** d_t,
                        double** d_y, double** d_u) {
    const int64_t ns = w.s1 - w.s0;
    int rc;
    if ((rc = upload(c, BUF_T, t + w.s0, ns, d_t))) return rc;
    if ((rc = upload(c, BUF_Y, y + w.s0, ns, d_y))) return rc;
    return upload(c, BUF_U, u ? u + w.s0 : nullptr, ns, d_u);
}
// the same for t and C channels of Y (channel c at Y + c ldY, on the device at *d_Y + c (s1 - s0)), Y scanned for NaN / Inf
static int upload_range_channels(lpvs_ctx* c, const Windows& w, const double* t, const double* Y, int C, int64_t ldY,
                                 double** d_t, double** d_Y) {
    const int64_t ns = w.s1 - w.s0;
    int rc;
    if ((rc = upload(c, BUF_T, t + w.s0, ns, d_t))) return rc;
    if ((rc = upload_channels(c, Y, C, ldY, w.s0, ns, d_Y))) return rc;
    scan_finite(c, *d_Y, (long long)C * ns);
    return LPVS_OK;
}

// lpvs_ls_window_sums[_dev] on device samples whose window 0 is window `base` of the caller's record
static int window_sums(lpvs_ctx* c, int kind, const double* d_y, const double* d_u, const double* d_t, int64_t N,
                       const double* f, int Nf, const double* W, int n, int noverlap, double lambda, int64_t k_begin,
                       int64_t k_end, int64_t base, double* sums, int* info) {
    cudaSetDevice(c->device);
    if (info) *info = 0;
    if (kind < 0 || kind > 2) return fail(c, LPVS_E_BAD_ARG, "bad window kind %d", kind);
    if (!d_y || !d_t || !W || !sums || n <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (kind != LPVS_WIN_PSD && !d_u) return fail(c, LPVS_E_BAD_ARG, "second signal required");
    Windows w;
    int rc = window_range(c, N, n, noverlap, k_begin, k_end, &w);
    if (rc) return rc;
    gram_timer_reset(c);
    FourierPlan pl;
    if ((rc = make_fourier_plan(c, f, Nf, &pl))) return rc;
    const int nrhs = kind == LPVS_WIN_PSD ? 1 : 2;
    const int slen = sums_len(kind, Nf);
    double* d_sums = ws<double>(c, BUF_SUMS, (size_t)slen);
    double* d_W;
    if ((rc = upload(c, BUF_W, W, n, &d_W))) return rc;
    if (!d_sums) return fail(c, LPVS_E_NOMEM, "out of device memory");
    LPVS_CU(c, cudaMemsetAsync(d_sums, 0, sizeof(double) * slen, c->st));
    const long long Np = pl.Np;
    // batch: the Gram workspace <= ~6 GiB
    const int64_t batch = batch_size(c, Np * Np * 8, 6LL << 30, true, INT64_MAX, k_end - k_begin);
    std::vector<int> hinfo((size_t)batch);
    FirstFailure bad;
    int jittered = 0;
    HostCopies copies{c->st};
    for (int64_t k0 = k_begin; k0 < k_end; k0 += batch) {
        const int nw = (int)std::min<int64_t>(batch, k_end - k0);
        double* d_G = ws<double>(c, BUF_G, (size_t)nw * Np * Np);
        double* d_B = ws<double>(c, BUF_B, (size_t)nw * 2 * Np);
        if (!d_G || !d_B) return fail(c, LPVS_E_NOMEM, "out of device memory (window batch of %d)", nw);
        GramArgs g;
        if ((rc = window_gram(c, pl, w, d_t, d_y, d_u, d_W, nrhs, k0, nw, false, true, d_G, d_B, g))) return rc;
        // always the weighted estimator: ridge lambda (src/lsfft.jl:121 -> :77)
        if ((rc = factor_solve(c, pl.Nf, pl.zero_first, pl.Np, d_G, d_B, nrhs, lambda, nw, hinfo.data()))) return rc;
        LPVS_CU(c, cudaStreamSynchronize(c->st));
        for (int i = 0; i < nw; i++) {
            if (hinfo[i] && c->jitter) {
                double* d_g1;
                if ((rc = jitter_refactor(c, pl, g, i, lambda, &d_g1, &hinfo[i]))) return rc;
                LPVS_CU(c, cudaMemcpyAsync(d_B + (long long)i * 2 * Np, d_g1 + Np * Np, sizeof(double) * 2 * Np,
                                           cudaMemcpyDeviceToDevice, c->st));
                LPVS_CU(c, cudaStreamSynchronize(c->st));
                jittered++;
            }
            bad.note(hinfo[i], base + k0 + i);
        }
        k_window_accum<<<(Nf + 127) / 128, 128, 0, c->st>>>(kind, d_B, 2 * Np, pl.Np, nw, Nf, pl.zero_first, d_sums);
        c->launches++;
    }
    copies.pending = false;
    LPVS_CU(c, cudaMemcpyAsync(sums, d_sums, sizeof(double) * slen, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    gram_timer_resolve(c);
    if (bad.pivot) return bad.report(c, info);
    if (jittered && info) *info = LPVS_INFO_JITTER;
    return LPVS_OK;
}

// ---- C channels at shared sample positions: per window ONE Gram matrix and ONE factor, C right-hand sides solved against it
// (k_gram_rhs_multi, k_trsm_multi), the C x C cross-spectral matrix accumulated on the device (k_window_matrix_accum).
// lpvs_ls_window_matrix_sums[_dev] on device samples whose window 0 is window `base` of the caller's record.
static int window_matrix_sums(lpvs_ctx* c, const double* d_Y, int C, int64_t ldY, const double* d_t, int64_t N,
                              const double* f, int Nf, const double* W, int n, int noverlap, double lambda,
                              int64_t k_begin, int64_t k_end, int64_t base, double* sums, int* info) {
    cudaSetDevice(c->device);
    if (info) *info = 0;
    if (C < 1) return fail(c, LPVS_E_BAD_ARG, "C must be >= 1 (got %d)", C);
    if (ldY < N) return fail(c, LPVS_E_BAD_ARG, "ldY (%lld) must be >= N (%lld)", (long long)ldY, (long long)N);
    if (!d_Y || !d_t || !W || !sums || n <= 0 || Nf <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    Windows w;
    int rc = window_range(c, N, n, noverlap, k_begin, k_end, &w);
    if (rc) return rc;
    gram_timer_reset(c);
    FourierPlan pl;
    if ((rc = make_fourier_plan(c, f, Nf, &pl))) return rc;
    const long long slen = 2LL * Nf * C * C;
    double* d_sums = ws<double>(c, BUF_SUMS, (size_t)slen);
    double* d_W;
    if ((rc = upload(c, BUF_W, W, n, &d_W))) return rc;
    if (!d_sums) return fail(c, LPVS_E_NOMEM, "out of device memory (%lld sums)", slen);
    LPVS_CU(c, cudaMemsetAsync(d_sums, 0, sizeof(double) * slen, c->st));
    const long long Np = pl.Np;
    const int nb = pl.Np / TB;
    // batch: Gram matrices, kept diagonal inverses and the C right-hand sides of a batch <= ~6 GiB
    const int64_t batch = batch_size(c, (Np * Np + Np * TB + (long long)C * Np) * 8, 6LL << 30, true, 32768, k_end - k_begin);
    std::vector<int> hinfo((size_t)batch);
    FirstFailure bad;
    int jittered = 0;
    HostCopies copies{c->st};
    for (int64_t k0 = k_begin; k0 < k_end; k0 += batch) {
        const int nw = (int)std::min<int64_t>(batch, k_end - k0);
        double* d_G = ws<double>(c, BUF_G, (size_t)nw * Np * Np);
        double* d_B = ws<double>(c, BUF_B, (size_t)nw * C * Np);
        if (!d_G || !d_B) return fail(c, LPVS_E_NOMEM, "out of device memory (window batch of %d, %d channels)", nw, C);
        GramArgs g;
        if ((rc = window_gram(c, pl, w, d_t, nullptr, nullptr, d_W, 0, k0, nw, true, true, d_G, nullptr, g))) return rc;
        // always the weighted estimator: ridge lambda (src/lsfft.jl:121 -> :77)
        if ((rc = factor_solve(c, pl.Nf, pl.zero_first, pl.Np, d_G, nullptr, 0, lambda, nw, hinfo.data()))) return rc;
        g.B = d_B;
        g.strideB = (long long)C * Np;
        c->launches += launch_gram_rhs_multi(pl.mode, g, d_Y, ldY, C, nw, c->st);
        CholArgs ca{};
        ca.G = d_G;
        ca.strideG = Np * Np;
        ca.Linv = ws<double>(c, BUF_LINV, (size_t)nw * nb * TB * TB);
        ca.strideLinv = (long long)nb * TB * TB;
        ca.info = ws<int>(c, BUF_INFO, (size_t)nw);
        ca.Np = pl.Np;
        ca.nb = nb;
        launch_trsm_multi(ca, d_B, (long long)C * Np, C, nw, c->st);
        c->launches++;
        LPVS_CU(c, cudaStreamSynchronize(c->st));
        for (int i = 0; i < nw; i++) {
            if (hinfo[i] && c->jitter) {
                // the window's C right-hand sides (left unsolved by k_trsm_multi) solved against its re-done factor
                double* d_g1;
                if ((rc = jitter_refactor(c, pl, g, i, lambda, &d_g1, &hinfo[i]))) return rc;
                CholArgs c1 = ca;
                c1.G = d_g1;
                launch_trsm_multi(c1, d_B + (long long)i * C * Np, (long long)C * Np, C, 1, c->st);
                c->launches++;
                LPVS_CU(c, cudaStreamSynchronize(c->st));
                jittered++;
            }
            bad.note(hinfo[i], base + k0 + i);
        }
        const long long nthr = (long long)Nf * C * C;
        k_window_matrix_accum<<<(unsigned)((nthr + 127) / 128), 128, 0, c->st>>>(d_B, (long long)C * Np, pl.Np, C, nw, Nf,
                                                                                 pl.zero_first, d_sums);
        c->launches++;
    }
    copies.pending = false;
    LPVS_CU(c, cudaMemcpyAsync(sums, d_sums, sizeof(double) * slen, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    gram_timer_resolve(c);
    if (bad.pivot) return bad.report(c, info);
    if (jittered && info) *info = LPVS_INFO_JITTER;
    return LPVS_OK;
}

}  // namespace lpvs

extern "C" {

int lpvs_ls_window_sums_dev(lpvs_ctx* c, int kind, const double* d_y, const double* d_u, const double* d_t,
                            int64_t N, const double* f, int Nf, const double* W, int n, int noverlap, double lambda,
                            int64_t k_begin, int64_t k_end, double* sums, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    return window_sums(c, kind, d_y, d_u, d_t, N, f, Nf, W, n, noverlap, lambda, k_begin, k_end, 0, sums, info);
}

int lpvs_ls_window_sums(lpvs_ctx* c, int kind, const double* y, const double* u, const double* t, int64_t N,
                        const double* f, int Nf, const double* W, int n, int noverlap, double lambda, int64_t k_begin,
                        int64_t k_end, double* sums, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);  // held across upload + compute: the uploaded samples live in the context's workspace
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (!y || !t || N <= 0 || n <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    Windows w;
    int rc = window_range(c, N, n, noverlap, k_begin, k_end, &w);
    if (rc) return rc;
    if (k_end == k_begin) {
        if (sums) memset(sums, 0, sizeof(double) * sums_len(kind, Nf));
        return LPVS_OK;
    }
    double *d_t, *d_y, *d_u;
    if ((rc = upload_range(c, w, t, y, u, &d_t, &d_y, &d_u))) return rc;
    const Windows r = w.uploaded();
    rc = window_sums(c, kind, d_y, d_u, d_t, r.N, f, Nf, W, n, noverlap, lambda, r.k_begin, r.k_end, k_begin, sums, info);
    const int rcf = inputs_finite(c);
    return rcf ? rcf : rc;
}

int lpvs_ls_window_matrix_sums_dev(lpvs_ctx* c, const double* d_Y, int C, int64_t ldY, const double* d_t, int64_t N,
                                   const double* f, int Nf, const double* W, int n, int noverlap, double lambda,
                                   int64_t k_begin, int64_t k_end, double* sums, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    return window_matrix_sums(c, d_Y, C, ldY, d_t, N, f, Nf, W, n, noverlap, lambda, k_begin, k_end, 0, sums, info);
}

int lpvs_ls_window_matrix_sums(lpvs_ctx* c, const double* Y, int C, int64_t ldY, const double* t, int64_t N,
                               const double* f, int Nf, const double* W, int n, int noverlap, double lambda,
                               int64_t k_begin, int64_t k_end, double* sums, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);  // held across upload + compute: the uploaded samples live in the context's workspace
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (info) *info = 0;
    if (C < 1) return fail(c, LPVS_E_BAD_ARG, "C must be >= 1 (got %d)", C);
    if (ldY < N) return fail(c, LPVS_E_BAD_ARG, "ldY (%lld) must be >= N (%lld)", (long long)ldY, (long long)N);
    if (!Y || !t || N <= 0 || n <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    Windows w;
    int rc = window_range(c, N, n, noverlap, k_begin, k_end, &w);
    if (rc) return rc;
    if (k_end == k_begin) {
        if (sums && Nf > 0) memset(sums, 0, sizeof(double) * 2 * (size_t)Nf * C * C);
        return LPVS_OK;
    }
    double *d_t, *d_Y;
    if ((rc = upload_range_channels(c, w, t, Y, C, ldY, &d_t, &d_Y))) return rc;
    const Windows r = w.uploaded();
    rc = window_matrix_sums(c, d_Y, C, r.N, d_t, r.N, f, Nf, W, n, noverlap, lambda, r.k_begin, r.k_end, k_begin, sums,
                            info);
    const int rcf = inputs_finite(c);
    return rcf ? rcf : rc;
}

int lpvs_ls_window_matrix_finalize(int kind, const double* sums, int Nf, int C, int64_t K, double* out) {
    if (!sums || !out || Nf <= 0 || C < 1) return LPVS_E_BAD_ARG;
    const long long CC = (long long)C * C;
    auto re = [&](int k, int i, int j) { return sums[2 * ((long long)k * CC + (long long)i * C + j)]; };
    auto im = [&](int k, int i, int j) { return sums[2 * ((long long)k * CC + (long long)i * C + j) + 1]; };
    if (kind == LPVS_WIN_PSD) {
        double k2 = (double)K * (double)K;  // S./nw^2  (src/lsfft.jl:125)
        for (int k = 0; k < Nf; k++)
            for (int i = 0; i < C; i++) out[(long long)k * C + i] = re(k, i, i) / k2;
    } else if (kind == LPVS_WIN_CSD) {
        double kk = (double)K;  // S./nw (src/lsfft.jl:155)
        for (long long e = 0; e < 2 * Nf * CC; e++) out[e] = sums[e] / kk;
    } else if (kind == LPVS_WIN_COHERE) {
        for (int k = 0; k < Nf; k++)  // abs2.(Syu)./(Suu.*Syy) (src/lsfft.jl:191) with y = channel i, u = channel j
            for (int i = 0; i < C; i++)
                for (int j = 0; j < C; j++) {
                    volatile double rr = re(k, i, j) * re(k, i, j);
                    volatile double ii = im(k, i, j) * im(k, i, j);
                    volatile double den = re(k, j, j) * re(k, i, i);
                    out[(long long)k * CC + (long long)i * C + j] = (rr + ii) / den;
                }
    } else {
        return LPVS_E_BAD_ARG;
    }
    return LPVS_OK;
}

}  // extern "C"

namespace lpvs {

// the arguments of the sparse windowed paths' ADMM
static int sparse_args(lpvs_ctx* c, int prox_kind, double mu) {
    if (!(mu > 0.0) || mu > 1.0) return fail(c, LPVS_E_BAD_ARG, "mu should be in (0, 1]");  // src/lasso.jl:143
    if (prox_kind < LPVS_PROX_L1 || prox_kind > LPVS_PROX_BALL_L0)
        return fail(c, LPVS_E_BAD_ARG, "prox kind %d not valid for the Fourier problem", prox_kind);
    return LPVS_OK;
}

// ---- C channels with estimator = ls_sparse_spectral: per window ONE inverse M = (A'WA + I/mu)^-1 (Gram and right-hand
// sides as window_matrix_sums, inverse as lpvs_ls_window_sparse_sums), every channel's ADMM once against it (k_admm_multi),
// the C x C matrix of the solutions accumulated by k_window_matrix_accum.
// lpvs_ls_window_matrix_sparse_sums[_dev] on device samples whose window 0 is window `base` of the caller's record.
static int window_matrix_sparse_sums(lpvs_ctx* c, const double* d_Y, int C, int64_t ldY, const double* d_t, int64_t N,
                                     const double* f, int Nf, const double* W, int n, int noverlap, int prox_kind,
                                     double prox_param, double mu, int64_t iters, double tol, int64_t k_begin,
                                     int64_t k_end, int64_t base, double* sums, int64_t* iters_done, double* residuals,
                                     int* info) {
    cudaSetDevice(c->device);
    if (info) *info = 0;
    if (C < 1) return fail(c, LPVS_E_BAD_ARG, "C must be >= 1 (got %d)", C);
    if (ldY < N) return fail(c, LPVS_E_BAD_ARG, "ldY (%lld) must be >= N (%lld)", (long long)ldY, (long long)N);
    if (N <= 0 || n <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    int rc = sparse_args(c, prox_kind, mu);
    if (rc) return rc;
    Windows w;
    if ((rc = window_range(c, N, n, noverlap, k_begin, k_end, &w))) return rc;
    if (!d_Y || !d_t || !W || !sums || Nf <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (C > 65535) return fail(c, LPVS_E_UNSUPPORTED, "C = %d channels: at most 65535", C);
    const long long slen = 2LL * Nf * C * C;
    if (k_end == k_begin) {
        memset(sums, 0, sizeof(double) * slen);
        return LPVS_OK;
    }
    gram_timer_reset(c);
    FourierPlan pl;
    if ((rc = make_fourier_plan(c, f, Nf, &pl))) return rc;
    double* d_sums = ws<double>(c, BUF_SUMS, (size_t)slen);
    double* d_W;
    if ((rc = upload(c, BUF_W, W, n, &d_W))) return rc;
    if (!d_sums) return fail(c, LPVS_E_NOMEM, "out of device memory (%lld sums)", slen);
    LPVS_CU(c, cudaMemsetAsync(d_sums, 0, sizeof(double) * slen, c->st));
    const long long Np = pl.Np;
    // batch: Gram/inverse, its workspace, kept diagonal inverses, the C right-hand sides and 7 Np of ADMM state per channel
    // <= ~6 GiB
    const int64_t batch =
        batch_size(c, (2 * Np * Np + Np * TB + 8LL * C * Np) * 8, 6LL << 30, true, 32768, k_end - k_begin);
    std::vector<int> hinfo((size_t)batch);
    std::vector<long long> hits((size_t)batch * C);
    long long* d_its = ws<long long>(c, BUF_WIN_ITS, (size_t)batch * C);
    double* d_res = ws<double>(c, BUF_WIN_RES, (size_t)batch * C);
    if (!d_its || !d_res) return fail(c, LPVS_E_NOMEM, "out of device memory (iteration counts)");
    FirstFailure bad;
    HostCopies copies{c->st};
    for (int64_t k0 = k_begin; k0 < k_end && !bad.pivot; k0 += batch) {
        const int nw = (int)std::min<int64_t>(batch, k_end - k0);
        double* d_G = ws<double>(c, BUF_G, (size_t)nw * Np * Np);
        double* d_Yi = ws<double>(c, BUF_YINV, (size_t)nw * Np * Np);
        double* d_B = ws<double>(c, BUF_B, (size_t)nw * C * Np);
        if (!d_G || !d_Yi || !d_B)
            return fail(c, LPVS_E_NOMEM, "out of device memory (window batch of %d, %d channels)", nw, C);
        GramArgs g;
        if ((rc = window_gram(c, pl, w, d_t, nullptr, nullptr, d_W, 0, k0, nw, true, true, d_G, nullptr, g))) return rc;
        if ((rc = batch_inverse(c, pl, d_G, d_Yi, nw, mu, hinfo.data()))) return rc;
        g.B = d_B;
        g.strideB = (long long)C * Np;
        c->launches += launch_gram_rhs_multi(pl.mode, g, d_Y, ldY, C, nw, c->st);
        if ((rc = admm_multi_run(c, d_G, d_B, pl.Np, C, nw, prox_kind, prox_param, mu, iters, tol, d_its, d_res, pl.Nf,
                                 pl.zero_first)))
            return rc;
        const long long nthr = (long long)Nf * C * C;
        k_window_matrix_accum<<<(unsigned)((nthr + 127) / 128), 128, 0, c->st>>>(d_B, (long long)C * Np, pl.Np, C, nw, Nf,
                                                                                 pl.zero_first, d_sums);
        c->launches++;
        const long long off = (k0 - k_begin) * C;
        if (iters_done) cudaMemcpyAsync(hits.data(), d_its, sizeof(long long) * nw * C, cudaMemcpyDeviceToHost, c->st);
        if (residuals)
            cudaMemcpyAsync(residuals + off, d_res, sizeof(double) * nw * C, cudaMemcpyDeviceToHost, c->st);
        cudaError_t e = cudaStreamSynchronize(c->st);
        if (e != cudaSuccess) return fail(c, LPVS_E_CUDA, "windowed sparse matrix batch failed: %s", cudaGetErrorString(e));
        if (iters_done)
            for (long long i = 0; i < (long long)nw * C; i++) iters_done[off + i] = hits[i];
        for (int i = 0; i < nw; i++) bad.note(hinfo[i], base + k0 + i);
    }
    copies.pending = false;
    if (bad.pivot) return bad.report(c, info);
    LPVS_CU(c, cudaMemcpyAsync(sums, d_sums, sizeof(double) * slen, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    gram_timer_resolve(c);
    return LPVS_OK;
}

}  // namespace lpvs

extern "C" {

// ---- windowed estimators with estimator = ls_sparse_spectral (src/lsfft.jl:121,150-151,184-185 calling the weighted
// method src/lasso.jl:105-126): every window is an independent ADMM problem on Quadratic(A'WA, A'Wy) (sign quirk Q13
// kept), x0 = 0.  Batched: Gram of all windows, batched Cholesky + SPD inverse of (A'WA + I/mu), then one CTA per
// window iterates to its own stop test (k_admm_batch); both channels of csd/cohere share the window's inverse.
int lpvs_ls_window_sparse_sums(lpvs_ctx* c, int kind, const double* y, const double* u, const double* t, int64_t N,
                               const double* f, int Nf, const double* W, int n, int noverlap, int prox_kind,
                               double prox_param, double mu, int64_t iters, double tol, int64_t k_begin,
                               int64_t k_end, double* sums, int64_t* iters_done, double* residuals, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (info) *info = 0;
    if (kind < 0 || kind > 2) return fail(c, LPVS_E_BAD_ARG, "bad window kind %d", kind);
    if (!y || !t || !W || !sums || N <= 0 || n <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (kind != LPVS_WIN_PSD && !u) return fail(c, LPVS_E_BAD_ARG, "second signal required");
    int rc = sparse_args(c, prox_kind, mu);
    if (rc) return rc;
    Windows w;
    if ((rc = window_range(c, N, n, noverlap, k_begin, k_end, &w))) return rc;
    const int nrhs = kind == LPVS_WIN_PSD ? 1 : 2;
    const int slen = sums_len(kind, Nf);
    if (k_end == k_begin) {
        memset(sums, 0, sizeof(double) * slen);
        return LPVS_OK;
    }
    gram_timer_reset(c);
    FourierPlan pl;
    if ((rc = make_fourier_plan(c, f, Nf, &pl))) return rc;
    double *d_t, *d_y, *d_u, *d_W;
    if ((rc = upload_range(c, w, t, y, u, &d_t, &d_y, &d_u))) return rc;
    if ((rc = upload(c, BUF_W, W, n, &d_W))) return rc;
    const Windows r = w.uploaded();
    double* d_sums = ws<double>(c, BUF_SUMS, (size_t)slen);
    if (!d_sums) return fail(c, LPVS_E_NOMEM, "out of device memory");
    LPVS_CU(c, cudaMemsetAsync(d_sums, 0, sizeof(double) * slen, c->st));
    const long long Np = pl.Np;
    // batch: Gram/inverse plus the inverse workspace <= ~6 GiB
    const int64_t batch = batch_size(c, Np * Np * 8, 3LL << 30, false, INT64_MAX, r.k_end);
    std::vector<int> hinfo((size_t)batch);
    std::vector<long long> hits((size_t)batch * nrhs);
    // per-window iteration counts and residuals live in the context's grow-only workspace (no allocation per call)
    long long* d_its = ws<long long>(c, BUF_WIN_ITS, (size_t)batch * nrhs);
    double* d_res = ws<double>(c, BUF_WIN_RES, (size_t)batch * nrhs);
    if (!d_its || !d_res) return fail(c, LPVS_E_NOMEM, "out of device memory");
    FirstFailure bad;
    HostCopies copies{c->st};
    for (int64_t k0 = 0; k0 < r.k_end && !bad.pivot; k0 += batch) {
        const int nw = (int)std::min<int64_t>(batch, r.k_end - k0);
        double* d_G = ws<double>(c, BUF_G, (size_t)nw * Np * Np);
        double* d_Y = ws<double>(c, BUF_YINV, (size_t)nw * Np * Np);
        double* d_B = ws<double>(c, BUF_B, (size_t)nw * 2 * Np);
        if (!d_G || !d_Y || !d_B) return fail(c, LPVS_E_NOMEM, "out of device memory (window batch of %d)", nw);
        // (the structured_ref correction is still scaled per batch here: its last bits depend on LPVS_OPT_WINDOW_BATCH)
        GramArgs g;
        if ((rc = window_gram(c, pl, r, d_t, d_y, d_u, d_W, nrhs, k0, nw, false, false, d_G, d_B, g))) return rc;
        if ((rc = batch_inverse(c, pl, d_G, d_Y, nw, mu, hinfo.data()))) return rc;
        if ((rc = admm_batch_run(c, d_G, d_B, pl.Np, nrhs, nw, prox_kind, prox_param, mu, /*quad=*/1, iters, tol, d_its,
                                 d_res, pl.Nf, pl.zero_first)))
            return rc;
        k_window_accum<<<(Nf + 127) / 128, 128, 0, c->st>>>(kind, d_B, 2 * Np, pl.Np, nw, Nf, pl.zero_first, d_sums);
        c->launches++;
        if (iters_done)
            cudaMemcpyAsync(hits.data(), d_its, sizeof(long long) * nw * nrhs, cudaMemcpyDeviceToHost, c->st);
        if (residuals)
            cudaMemcpyAsync(residuals + k0 * nrhs, d_res, sizeof(double) * nw * nrhs, cudaMemcpyDeviceToHost, c->st);
        cudaError_t e = cudaStreamSynchronize(c->st);
        if (e != cudaSuccess) return fail(c, LPVS_E_CUDA, "windowed sparse batch failed: %s", cudaGetErrorString(e));
        if (iters_done)
            for (int i = 0; i < nw * nrhs; i++) iters_done[k0 * nrhs + i] = hits[i];
        for (int i = 0; i < nw; i++) bad.note(hinfo[i], k_begin + k0 + i);
    }
    copies.pending = false;
    // a NaN / Inf input is reported ahead of a breakdown it may have caused, and leaves sums and info untouched
    if ((rc = inputs_finite(c))) return rc;
    if (bad.pivot) return bad.report(c, info);
    LPVS_CU(c, cudaMemcpyAsync(sums, d_sums, sizeof(double) * slen, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    gram_timer_resolve(c);
    return LPVS_OK;
}

int lpvs_ls_window_matrix_sparse_sums_dev(lpvs_ctx* c, const double* d_Y, int C, int64_t ldY, const double* d_t,
                                          int64_t N, const double* f, int Nf, const double* W, int n, int noverlap,
                                          int prox_kind, double prox_param, double mu, int64_t iters, double tol,
                                          int64_t k_begin, int64_t k_end, double* sums, int64_t* iters_done,
                                          double* residuals, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    return window_matrix_sparse_sums(c, d_Y, C, ldY, d_t, N, f, Nf, W, n, noverlap, prox_kind, prox_param, mu, iters, tol,
                                     k_begin, k_end, 0, sums, iters_done, residuals, info);
}

int lpvs_ls_window_matrix_sparse_sums(lpvs_ctx* c, const double* Y, int C, int64_t ldY, const double* t, int64_t N,
                                      const double* f, int Nf, const double* W, int n, int noverlap, int prox_kind,
                                      double prox_param, double mu, int64_t iters, double tol, int64_t k_begin,
                                      int64_t k_end, double* sums, int64_t* iters_done, double* residuals, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);  // held across upload + compute: the uploaded samples live in the context's workspace
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (info) *info = 0;
    if (C < 1) return fail(c, LPVS_E_BAD_ARG, "C must be >= 1 (got %d)", C);
    if (ldY < N) return fail(c, LPVS_E_BAD_ARG, "ldY (%lld) must be >= N (%lld)", (long long)ldY, (long long)N);
    if (N <= 0 || n <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    int rc = sparse_args(c, prox_kind, mu);
    if (rc) return rc;
    Windows w;
    if ((rc = window_range(c, N, n, noverlap, k_begin, k_end, &w))) return rc;
    if (!Y || !t || !sums || Nf <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (k_end == k_begin) {
        memset(sums, 0, sizeof(double) * 2 * (size_t)Nf * C * C);
        return LPVS_OK;
    }
    double *d_t, *d_Y;
    if ((rc = upload_range_channels(c, w, t, Y, C, ldY, &d_t, &d_Y))) return rc;
    const Windows r = w.uploaded();
    rc = window_matrix_sparse_sums(c, d_Y, C, r.N, d_t, r.N, f, Nf, W, n, noverlap, prox_kind, prox_param, mu, iters, tol,
                                   r.k_begin, r.k_end, k_begin, sums, iters_done, residuals, info);
    const int rcf = inputs_finite(c);
    return rcf ? rcf : rc;
}

int lpvs_ls_window_finalize(int kind, const double* sums, int Nf, int64_t K, double* out) {
    if (!sums || !out || Nf <= 0) return LPVS_E_BAD_ARG;
    if (kind == LPVS_WIN_PSD) {
        double k2 = (double)K * (double)K;  // S./nw^2  (src/lsfft.jl:125)
        for (int k = 0; k < Nf; k++) out[k] = sums[k] / k2;
    } else if (kind == LPVS_WIN_CSD) {
        double kk = (double)K;  // S./nw (src/lsfft.jl:155)
        for (int k = 0; k < Nf; k++) {
            out[2 * k] = sums[k] / kk;
            out[2 * k + 1] = sums[Nf + k] / kk;
        }
    } else if (kind == LPVS_WIN_COHERE) {
        for (int k = 0; k < Nf; k++) {  // abs2.(Syu)./(Suu.*Syy) (src/lsfft.jl:191)
            volatile double rr = sums[2 * Nf + k] * sums[2 * Nf + k];
            volatile double ii = sums[3 * Nf + k] * sums[3 * Nf + k];
            volatile double den = sums[Nf + k] * sums[k];
            out[k] = (rr + ii) / den;
        }
    } else {
        return LPVS_E_BAD_ARG;
    }
    return LPVS_OK;
}

int lpvs_ls_window(lpvs_ctx* c, int kind, const double* y, const double* u, const double* t, int64_t N,
                   const double* f, int Nf, const double* W, int n, int noverlap, double lambda, double* out,
                   int64_t* Kout, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    if (n <= 0 || Nf <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    int64_t K = lpvs_window_count(N, n, noverlap);
    if (K < 0) return fail(c, LPVS_E_BAD_ARG, "noverlap must be < n");
    if (Kout) *Kout = K;
    std::vector<double> sums((size_t)sums_len(kind, Nf), 0.0);
    if (K > 0) {
        int rc = lpvs_ls_window_sums(c, kind, y, u, t, N, f, Nf, W, n, noverlap, lambda, 0, K, sums.data(), info);
        if (rc) return rc;
    }
    return lpvs_ls_window_finalize(kind, sums.data(), Nf, K, out);
}

}  // extern "C"
