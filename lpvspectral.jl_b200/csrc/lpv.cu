// LPV (Fourier x RBF) estimators, ADMM problem construction and the row-sharded Gram entry points.
#include <math.h>

#include <algorithm>
#include <vector>

#include "ctx.h"

namespace lpvs {

namespace {

// e_n = sum_cc Re(A[n,cc]) p_re[cc] + Im(A[n,cc]) p_im[cc] - Y_n   (src/lsfft.jl:252: AA*real_params - Y)
__global__ void k_lpv_residual(const double2* __restrict__ E, const double* __restrict__ Kt, long long N, int Nf,
                               int Nvv, const double* __restrict__ xint, const double* __restrict__ Y,
                               double* __restrict__ e) {
    long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= N) return;
    double acc = 0.0;
    for (int k = 0; k < Nvv; k++) {
        double kv = Kt[(long long)k * N + s];
        double part = 0.0;
        for (int f = 0; f < Nf; f++) {
            int cc = f + k * Nf;
            int p = (cc >> 6) * 128 + (cc & 63);
            double2 ev = E[(long long)f * N + s];
            part = fma(ev.x, xint[p], part);
            part = fma(ev.y, xint[p + 64], part);
        }
        acc = fma(kv, part, acc);
    }
    e[s] = acc - Y[s];
}

// S[c][f] += abs2(sum_k X[c][f + k Nf]) for channel c = blockIdx.y   (psd(::SpectralExt), src/lsfft.jl:214-217, accumulated
// as src/lsfft.jl:273-274)
__global__ void k_lpv_psd_accum_multi(const double* __restrict__ X, long long ldx, int Nf, int Nvv, double* __restrict__ S) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= Nf) return;
    const double* xint = X + (long long)blockIdx.y * ldx;
    double re = 0.0, im = 0.0;
    for (int k = 0; k < Nvv; k++) {
        const int cc = f + k * Nf;
        const int p = (cc >> 6) * 128 + (cc & 63);
        re += xint[p];
        im += xint[p + 64];
    }
    double* s = S + (long long)blockIdx.y * Nf + f;
    *s = __dadd_rn(*s, __dadd_rn(__dmul_rn(re, re), __dmul_rn(im, im)));
}

// block partial sums of (v - shift[c]) and (v - shift[c])^2 for channel c = blockIdx.y of v (ld ldv; shift null: 0):
// partials out[c][block][2]
__global__ void k_sum_sq_multi(const double* __restrict__ v, long long ldv, long long N, const double* __restrict__ shift,
                               double* __restrict__ out) {
    __shared__ double s1[256], s2[256];
    const int ch = blockIdx.y;
    const double* vc = v + ch * ldv;
    const double sh = shift ? shift[ch] : 0.0;
    double a = 0.0, b = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        double d = vc[i] - sh;
        a += d;
        b += d * d;
    }
    s1[threadIdx.x] = a;
    s2[threadIdx.x] = b;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            s1[threadIdx.x] += s1[threadIdx.x + s];
            s2[threadIdx.x] += s2[threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[((long long)ch * gridDim.x + blockIdx.x) * 2] = s1[0];
        out[((long long)ch * gridDim.x + blockIdx.x) * 2 + 1] = s2[0];
    }
}

// one thread per channel: the nb block partials [which] summed in block order, / den
__global__ void k_sum_parts_multi(const double* __restrict__ part, int nb, int which, double den, int C,
                                  double* __restrict__ out) {
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= C) return;
    double s = 0.0;
    for (int i = 0; i < nb; i++) s += part[((long long)ch * nb + i) * 2 + which];
    out[ch] = s / den;
}

__global__ void k_scale(double* v, long long n, double s) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] *= s;
}

// var(v) with n-1 (Julia `var`) of C channels (channel c at d_v + c ldv), two passes on device in one launch each; the block
// partials of a channel are summed in fixed order, so its variance does not depend on C; d_var: C doubles on the device
int device_var_multi(lpvs_ctx* c, const double* d_v, long long ldv, long long N, int C, double* d_var) {
    const int nb = 256;
    double* d_p = ws<double>(c, BUF_SUMS, (size_t)2 * nb * C + C);
    if (!d_p) return fail(c, LPVS_E_NOMEM, "out of device memory (variances of %d channels)", C);
    double* d_mean = d_p + 2LL * nb * C;
    const unsigned gc = (unsigned)((C + 127) / 128);
    k_sum_sq_multi<<<dim3(nb, C), 256, 0, c->st>>>(d_v, ldv, N, nullptr, d_p);
    k_sum_parts_multi<<<gc, 128, 0, c->st>>>(d_p, nb, 0, (double)N, C, d_mean);
    k_sum_sq_multi<<<dim3(nb, C), 256, 0, c->st>>>(d_v, ldv, N, d_mean, d_p);
    k_sum_parts_multi<<<gc, 128, 0, c->st>>>(d_p, nb, 1, (double)(N - 1), C, d_var);
    c->launches += 4;
    LPVS_CU(c, cudaGetLastError());
    return LPVS_OK;
}

}  // namespace

// tables for samples [0,N) of DEVICE arrays d_X / d_V; V is the same range on the HOST (centres need its min / max)
int lpv_prepare_dev(lpvs_ctx* c, const double* V, const double* d_X, const double* d_V, int64_t N, const double* d_w,
                    int Nf, int Nv, int coulomb, int normalize, LpvPlan* pl) {
    pl->Nf = Nf;
    pl->Nv = Nv;
    pl->Nvv = coulomb ? 2 * Nv : Nv;
    pl->ncc = Nf * pl->Nvv;
    pl->nblk = (pl->ncc + FB - 1) / FB;
    pl->Np = pl->nblk * TB;
    pl->coulomb = coulomb;
    pl->normalize = normalize;
    pl->N = N;
    // basis_activation_func (src/utilities.jl:23-36): centres and gamma on the host (O(N) min/max)
    std::vector<double> cen((size_t)pl->Nvv);
    double gamma;
    if (coulomb) {
        double m = 0.0;
        for (int64_t i = 0; i < N; i++) m = std::max(m, fabs(V[i]));
        int num = Nv + 2;
        double step = m / (double)(num - 1);
        std::vector<double> vc((size_t)Nv);
        for (int k = 0; k < Nv; k++) vc[k] = (k + 1) * step;  // range(0, m, Nv+2)[2:end-1]
        for (int k = 0; k < Nv; k++) {
            cen[k] = -vc[Nv - 1 - k];
            cen[Nv + k] = vc[k];
        }
        gamma = (double)pl->Nvv / fabs(cen[0] - cen[pl->Nvv - 1]);
    } else {
        double lo = V[0], hi = V[0];
        for (int64_t i = 1; i < N; i++) {
            lo = std::min(lo, V[i]);
            hi = std::max(hi, V[i]);
        }
        if (Nv == 1) {
            cen[0] = lo;
        } else {
            double step = (hi - lo) / (double)(Nv - 1);
            for (int k = 0; k < Nv; k++) cen[k] = lo + k * step;
            cen[Nv - 1] = hi;
        }
        gamma = (double)Nv / fabs(cen[0] - cen[Nv - 1]);
    }
    if (!isfinite(gamma)) return fail(c, LPVS_E_BAD_ARG, "degenerate scheduling signal (all V equal)");
    double* d_cen;
    int rc;
    if ((rc = upload(c, BUF_CENT, cen.data(), pl->Nvv, &d_cen))) return rc;
    double2* E = ws<double2>(c, BUF_E, (size_t)Nf * N);
    double* K = ws<double>(c, BUF_K, (size_t)pl->Nvv * N);
    if (!E || !K) return fail(c, LPVS_E_NOMEM, "out of device memory (LPV tables)");
    launch_lpv_tables(d_X, d_V, N, d_w, Nf, pl->Nvv, d_cen, gamma, coulomb, normalize, E, K, c->d_nonfinite, c->st);
    c->launches++;
    pl->d_E = E;
    pl->d_K = K;
    return LPVS_OK;
}

int lpv_prepare(lpvs_ctx* c, const double* X, const double* V, int64_t N, const double* w, int Nf, int Nv,
                int coulomb, int normalize, LpvPlan* pl) {
    if (!X || !V || !w || N <= 1 || Nf <= 0 || Nv <= 0) return fail(c, LPVS_E_BAD_ARG, "bad LPV arguments");
    double *d_X, *d_V, *d_w;
    int rc;
    if ((rc = upload(c, BUF_T, X, N, &d_X))) return rc;
    if ((rc = upload(c, BUF_V, V, N, &d_V))) return rc;
    if ((rc = upload(c, BUF_F, w, Nf, &d_w))) return rc;
    return lpv_prepare_dev(c, V, d_X, d_V, N, d_w, Nf, Nv, coulomb, normalize, pl);
}

int lpv_gram(lpvs_ctx* c, const LpvPlan& pl, const double* d_y, double* d_G, double* d_B) {
    const long long Np = pl.Np;
    const int ntiles = pl.nblk * (pl.nblk + 1) / 2;
    int nsplit = 1;
    if (ntiles < 4 * c->sms) {
        long long want = (4LL * c->sms + ntiles - 1) / ntiles;
        long long maxs = std::max<long long>(1, pl.N / 2048);
        nsplit = (int)std::min(want, maxs);
    }
    GramArgs g{};
    g.t = nullptr;
    g.y = d_y;
    g.u = nullptr;
    g.W = nullptr;
    g.w_abs = 1;
    g.ncc = pl.ncc;
    g.nblk = pl.nblk;
    g.nrhs = d_y ? 1 : 0;
    g.tbl_base = 0;
    g.tbl_ns = pl.N;
    g.E = pl.d_E;
    g.Kt = pl.d_K;
    g.lpv_nf = pl.Nf;
    g.gscale = 1.0;
    g.bscale = 1.0;
    g.s_end = pl.N;
    long long n_split = (pl.N + nsplit - 1) / nsplit;
    n_split = (n_split + KC - 1) / KC * KC;
    int nprob = (int)((pl.N + n_split - 1) / n_split);
    g.start0 = 0;
    g.hop = n_split;
    g.n = (int)n_split;
    const long long part_stride = Np * Np + 2 * Np;
    double* parts = nullptr;
    if (nprob == 1) {
        g.G = d_G;
        g.B = d_B;
    } else {
        parts = ws<double>(c, BUF_PART, (size_t)nprob * part_stride);
        if (!parts) return fail(c, LPVS_E_NOMEM, "out of device memory (Gram partials)");
        g.G = parts;
        g.strideG = part_stride;
        g.B = parts + Np * Np;
        g.strideB = part_stride;
    }
    gram_timer_begin(c);
    c->launches += launch_gram(GRAM_LPV, g, nprob, c->st);
    gram_timer_end(c, (double)pl.N * (2.0 * pl.ncc) * (2.0 * pl.ncc + 1.0), 1);
    if (nprob > 1) {
        reduce_parts(c, d_G, parts, Np * Np, part_stride, nprob, 0);
        if (d_B) reduce_parts(c, d_B, parts + Np * Np, 2 * Np, part_stride, nprob, 0);
    }
    LPVS_CU(c, cudaGetLastError());
    return LPVS_OK;
}

}  // namespace lpvs

namespace lpvs {
namespace {

// inv(Ar'Ar + lambda I) (src/lsfft.jl:254) into d_out (nref x nref, reference column order) from the second copy of G at
// d_G + Np^2; the first copy (holding the solve's factor) serves as the inverse workspace.  *pinfo: the breakdown pivot.
int lpv_sigma_inverse(lpvs_ctx* c, const LpvPlan& pl, double* d_G, double lambda, double* d_out, int* pinfo) {
    const long long NN = (long long)pl.Np * pl.Np;
    double* d_G2 = d_G + NN;
    CholArgs ca{};
    ca.G = d_G2;
    ca.strideG = NN;
    ca.Y = d_G;
    ca.strideY = NN;
    ca.Linv = ws<double>(c, BUF_LINV, (size_t)pl.nblk * TB * TB);
    ca.strideLinv = (long long)pl.nblk * TB * TB;
    ca.info = ws<int>(c, BUF_INFO, 1);
    ca.Np = pl.Np;
    ca.nb = pl.nblk;
    LPVS_CU(c, cudaMemsetAsync(ca.info, 0, sizeof(int), c->st));
    launch_diag_prepare(d_G2, NN, pl.Np, pl.ncc, 0, nullptr, lambda, 1, c->st);
    c->launches += 1 + potrf(ca, 1, c->sms, c->st, &c->la);
    LPVS_CU(c, cudaMemcpyAsync(pinfo, ca.info, sizeof(int), cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    if (*pinfo) return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown (Sigma) at internal pivot %d", *pinfo);
    c->launches += potri(ca, 1, c->st);
    launch_gather_ref(c, d_G2, nullptr, pl.Np, pl.ncc, 0, 2 * pl.ncc, d_out, nullptr);
    return LPVS_OK;
}

// the LPV regressor of a plan as an operator (lsq.cu)
OpArgs lpv_op(const LpvPlan& pl) {
    OpArgs op;
    op.mode = GRAM_LPV;
    op.E = pl.d_E;
    op.Kt = pl.d_K;
    op.tbl_ns = pl.N;
    op.lpv_nf = pl.Nf;
    op.ncc = pl.ncc;
    op.zero_first = 0;
    op.N = pl.N;
    return op;
}

// ls_spectral_lpv on prepared tables and a device-resident Y (src/lsfft.jl:248-257); params / Sigma / fva are host outputs
// params (host, nullable) and / or d_psd (device, nullable: S[f] += abs2(sum_k x[f,k]) stays on the device)
int lpv_ls_core(lpvs_ctx* c, const LpvPlan& pl, const double* d_Y, double lambda, double* params, double* Sigma,
                double* fva, int* info, double* d_psd = nullptr) {
    const int64_t N = pl.N;
    const int Nf = pl.Nf;
    int rc;
    const long long Np = pl.Np, NN = Np * Np;
    const int nref = 2 * pl.ncc;
    // two copies of G: ridge lambda^2 for the solve (src/utilities.jl:52), ridge lambda for Sigma (src/lsfft.jl:254)
    double* d_G = ws<double>(c, BUF_G, (size_t)(Sigma ? 2 : 1) * NN);
    double* d_B = ws<double>(c, BUF_B, (size_t)2 * Np);
    if (!d_G || !d_B) return fail(c, LPVS_E_NOMEM, "out of device memory (G)");
    if ((rc = lpv_gram(c, pl, d_Y, d_G, d_B))) return rc;
    if (Sigma) LPVS_CU(c, cudaMemcpyAsync(d_G + NN, d_G, sizeof(double) * NN, cudaMemcpyDeviceToDevice, c->st));
    int pinfo = 0;
    if (c->jitter) {
        // the reference solves on [Ar; lambda I] itself (pivoted QR, src/utilities.jl:52): operator-accurate solve, so the
        // default lambda = 1e-8 (ridge 1e-16, far below what a Cholesky of the Gram matrix can resolve) works
        auto regram = [&]() { return lpv_gram(c, pl, d_Y, d_G, d_B); };
        rc = ls_solve_accurate(c, lpv_op(pl), pl.Np, 0, d_Y, d_G, d_B, lambda, regram, info);
        if (rc) {
            const int rcf = inputs_finite(c);  // NaN inputs / 0/0 basis normalisation: the cause, not "not SPD"
            return rcf ? rcf : rc;
        }
    } else {
        if ((rc = factor_solve(c, pl.ncc, 0, pl.Np, d_G, d_B, 1, lambda * lambda, 1, &pinfo))) return rc;
        if ((rc = inputs_finite(c))) return rc;
        LPVS_CU(c, cudaStreamSynchronize(c->st));
        if (pinfo) {
            if (info) *info = pinfo;
            return fail(c, LPVS_E_NOT_SPD,
                        "Cholesky breakdown at internal pivot %d: Ar'Ar + lambda^2 I is not numerically positive definite "
                        "(lambda=%g; LPVS_OPT_JITTER=0 disabled the QR-class solve)", pinfo, lambda);
        }
    }
    double* d_out = ws<double>(c, BUF_X, (size_t)nref);
    double* d_e = ws<double>(c, BUF_MISC, (size_t)std::max<long long>(N, (long long)nref * nref));
    if (!d_out || !d_e) return fail(c, LPVS_E_NOMEM, "out of device memory");
    if (params) {
        launch_x_to_complex(c, d_B, pl.Np, pl.ncc, 0, 1, d_out);
        LPVS_CU(c, cudaMemcpyAsync(params, d_out, sizeof(double) * nref, cudaMemcpyDeviceToHost, c->st));
    }
    if (d_psd) {
        k_lpv_psd_accum_multi<<<dim3((Nf + 127) / 128, 1), 128, 0, c->st>>>(d_B, Np, Nf, pl.Nvv, d_psd);
        c->launches++;
    }
    // residual, variances, fraction of variance explained (src/lsfft.jl:252-256)
    double hv[2] = {0.0, 0.0};  // var(e), var(y)
    if (fva || Sigma) {
        double* d_v = ws<double>(c, BUF_MC_NRM, 2);
        if (!d_v) return fail(c, LPVS_E_NOMEM, "out of device memory");
        k_lpv_residual<<<(unsigned)((N + 127) / 128), 128, 0, c->st>>>(pl.d_E, pl.d_K, N, Nf, pl.Nvv, d_B, d_Y, d_e);
        c->launches++;
        if ((rc = device_var_multi(c, d_e, N, N, 1, d_v))) return rc;
        if (fva && (rc = device_var_multi(c, d_Y, N, N, 1, d_v + 1))) return rc;
        LPVS_CU(c, cudaMemcpyAsync(hv, d_v, sizeof(double) * (fva ? 2 : 1), cudaMemcpyDeviceToHost, c->st));
        LPVS_CU(c, cudaStreamSynchronize(c->st));
    }
    if (fva) *fva = 1.0 - hv[0] / hv[1];
    if (Sigma) {
        if ((rc = lpv_sigma_inverse(c, pl, d_G, lambda, d_e, &pinfo))) {
            if (pinfo && info) *info = pinfo;
            return rc;
        }
        k_scale<<<(unsigned)(((long long)nref * nref + 255) / 256), 256, 0, c->st>>>(d_e, (long long)nref * nref, hv[0]);
        c->launches++;
        LPVS_CU(c, cudaMemcpyAsync(Sigma, d_e, sizeof(double) * nref * nref, cudaMemcpyDeviceToHost, c->st));
    }
    return inputs_finite(c);
}

// lpv_ls_core for C channels (channel c at d_Y + c ldY) on one set of tables: the Gram matrix, its factors and Sigma0 =
// inv(Ar'Ar + lambda I) are built once; the solve runs C-wide (ls_solve_accurate_multi).  Host outputs (all nullable):
// params [C][2 ncc], Sigma0, var_e [C], fva [C]; info [C]; d_psd [C][Nf] accumulates on the device.
int lpv_ls_core_multi(lpvs_ctx* c, const LpvPlan& pl, const double* d_Y, long long ldY, int C, double lambda,
                      double* params, double* Sigma0, double* var_e, double* fva, int* info, double* d_psd) {
    const int64_t N = pl.N;
    const int Nf = pl.Nf;
    int rc;
    const long long Np = pl.Np, NN = Np * Np;
    const int nref = 2 * pl.ncc;
    for (int ch = 0; ch < C; ch++) info[ch] = 0;
    // two copies of G, as lpv_ls_core: ridge lambda^2 for the solve, ridge lambda for Sigma0
    double* d_G = ws<double>(c, BUF_G, (size_t)(Sigma0 ? 2 : 1) * NN);
    double* d_Bs = ws<double>(c, BUF_B, (size_t)2 * Np);
    double* d_X = ws<double>(c, BUF_MC_X, (size_t)C * Np);
    if (!d_G || !d_Bs || !d_X) return fail(c, LPVS_E_NOMEM, "out of device memory (G, %d channels)", C);
    // G only: the right-hand sides are formed C-wide by the solve
    auto regram = [&]() { return lpv_gram(c, pl, nullptr, d_G, d_Bs); };
    if ((rc = regram())) return rc;
    if (Sigma0) LPVS_CU(c, cudaMemcpyAsync(d_G + NN, d_G, sizeof(double) * NN, cudaMemcpyDeviceToDevice, c->st));
    const OpArgs op = lpv_op(pl);
    if (c->jitter) {
        if ((rc = ls_solve_accurate_multi(c, op, pl.Np, 0, d_Y, ldY, C, d_G, lambda, regram, d_X, info))) {
            const int rcf = inputs_finite(c);  // NaN inputs / 0/0 basis normalisation: the cause, not "not SPD"
            return rcf ? rcf : rc;
        }
    } else {
        // one plain Cholesky of Ar'Ar + lambda^2 I, C solves through the explicit inverse factor
        int pinfo = 0;
        if ((rc = factor_solve(c, pl.ncc, 0, pl.Np, d_G, nullptr, 0, lambda * lambda, 1, &pinfo))) return rc;
        if ((rc = inputs_finite(c))) return rc;
        if (pinfo) {
            for (int ch = 0; ch < C; ch++) info[ch] = pinfo;
            return fail(c, LPVS_E_NOT_SPD,
                        "Cholesky breakdown at internal pivot %d: Ar'Ar + lambda^2 I is not numerically positive definite "
                        "(lambda=%g; LPVS_OPT_JITTER=0 disabled the QR-class solve)", pinfo, lambda);
        }
        GramArgs g{};
        g.w_abs = 1;
        g.s_end = N;
        g.ncc = pl.ncc;
        g.nblk = pl.nblk;
        g.tbl_ns = N;
        g.E = pl.d_E;
        g.Kt = pl.d_K;
        g.lpv_nf = Nf;
        g.gscale = 1.0;
        g.bscale = 1.0;
        if ((rc = chol_solve_multi(c, g, GRAM_LPV, pl.Np, d_G, d_Y, ldY, C, d_X))) return rc;
    }
    if (params) {
        double* d_out = ws<double>(c, BUF_X, (size_t)nref * C);
        if (!d_out) return fail(c, LPVS_E_NOMEM, "out of device memory (params of %d channels)", C);
        launch_x_to_complex(c, d_X, pl.Np, pl.ncc, 0, C, d_out);
        LPVS_CU(c, cudaMemcpyAsync(params, d_out, sizeof(double) * nref * C, cudaMemcpyDeviceToHost, c->st));
    }
    if (d_psd) {
        k_lpv_psd_accum_multi<<<dim3((Nf + 127) / 128, C), 128, 0, c->st>>>(d_X, Np, Nf, pl.Nvv, d_psd);
        c->launches++;
    }
    // residuals R = Y - Ar x (the variance does not depend on the sign), variances, fraction of variance explained
    if (fva || var_e) {
        double* d_R = ws<double>(c, BUF_MC_W, (size_t)C * N);
        double* d_v = ws<double>(c, BUF_MC_NRM, (size_t)2 * C);  // var(e) | var(y)
        if (!d_R || !d_v) return fail(c, LPVS_E_NOMEM, "out of device memory (residuals of %d channels)", C);
        op_residual_multi(c, op, d_X, pl.Np, d_Y, ldY, d_R, N, C);
        if ((rc = device_var_multi(c, d_R, N, N, C, d_v))) return rc;
        if (fva && (rc = device_var_multi(c, d_Y, ldY, N, C, d_v + C))) return rc;
        std::vector<double> hv((size_t)2 * C);
        LPVS_CU(c, cudaMemcpyAsync(hv.data(), d_v, sizeof(double) * (fva ? 2 : 1) * C, cudaMemcpyDeviceToHost, c->st));
        LPVS_CU(c, cudaStreamSynchronize(c->st));
        for (int ch = 0; ch < C; ch++) {
            if (var_e) var_e[ch] = hv[ch];
            if (fva) fva[ch] = 1.0 - hv[ch] / hv[C + ch];
        }
    }
    if (Sigma0) {
        double* d_e = ws<double>(c, BUF_MISC, (size_t)nref * nref);
        if (!d_e) return fail(c, LPVS_E_NOMEM, "out of device memory (Sigma)");
        int pinfo = 0;
        if ((rc = lpv_sigma_inverse(c, pl, d_G, lambda, d_e, &pinfo))) {
            if (pinfo)
                for (int ch = 0; ch < C; ch++) info[ch] = pinfo;
            return rc;
        }
        LPVS_CU(c, cudaMemcpyAsync(Sigma0, d_e, sizeof(double) * nref * nref, cudaMemcpyDeviceToHost, c->st));
    }
    return inputs_finite(c);
}

// LPVS_E_NONFINITE naming the first of the C device channels that holds a NaN or Inf
int check_channels_finite(lpvs_ctx* c, const double* d_Y, long long ldY, long long N, int C) {
    int* d_flag = ws<int>(c, BUF_MC_ACT, (size_t)C);
    if (!d_flag) return fail(c, LPVS_E_NOMEM, "out of device memory (flags)");
    int h = C;
    LPVS_CU(c, cudaMemcpyAsync(d_flag, &h, sizeof h, cudaMemcpyHostToDevice, c->st));
    const unsigned nblk = (unsigned)std::min<long long>((N + 255) / 256, 64);
    k_first_nonfinite_channel<<<dim3(nblk, C), 256, 0, c->st>>>(d_Y, ldY, N, d_flag);
    c->launches++;
    LPVS_CU(c, cudaMemcpyAsync(&h, d_flag, sizeof h, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    if (h < C) return fail(c, LPVS_E_NONFINITE, "non-finite value (NaN/Inf) in channel %d", h);
    return LPVS_OK;
}

}  // namespace
}  // namespace lpvs

using namespace lpvs;

extern "C" {

int lpvs_ls_spectral_lpv(lpvs_ctx* c, const double* Y, const double* X, const double* V, int64_t N, const double* w,
                         int Nf, int Nv, double lambda, int coulomb, int normalize, double* params, double* Sigma,
                         double* fva, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (info) *info = 0;
    if (!Y || !params) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    gram_timer_reset(c);
    LpvPlan pl;
    int rc = lpv_prepare(c, X, V, N, w, Nf, Nv, coulomb, normalize, &pl);
    if (rc) return rc;
    double* d_Y;
    if ((rc = upload(c, BUF_Y, Y, N, &d_Y))) return rc;
    if ((rc = lpv_ls_core(c, pl, d_Y, lambda, params, Sigma, fva, info))) return rc;
    gram_timer_resolve(c);
    return LPVS_OK;
}

// ls_windowpsd_lpv (src/lsfft.jl:267-277): Y, X, V, w go to the device once; every rect window (Windows3,
// src/windows.jl:94-104) is a sample range of those arrays with its own basis centres (basis_activation_func is
// evaluated on the window's V) and runs the dense LPV estimator above.
int lpvs_ls_windowpsd_lpv(lpvs_ctx* c, const double* Y, const double* X, const double* V, int64_t N, const double* w,
                          int Nf, int Nv, int n, int noverlap, double lambda, int coulomb, int normalize, double* S,
                          double* fva, int64_t* K, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (info) *info = 0;
    if (K) *K = 0;
    if (!Y || !X || !V || !w || !S || N <= 0 || Nf <= 0 || Nv <= 0 || n <= 1)
        return fail(c, LPVS_E_BAD_ARG, "bad LPV window arguments");
    if (noverlap < 0) noverlap = n >> 1;  // src/windows.jl:97
    if (noverlap >= n) return fail(c, LPVS_E_BAD_ARG, "noverlap must be smaller than the window length");
    const int64_t hop = n - noverlap;
    const int64_t nwin = N >= n ? (N - n) / hop + 1 : 0;
    if (K) *K = nwin;
    for (int f = 0; f < Nf; f++) S[f] = 0.0;
    if (nwin == 0) return LPVS_OK;
    gram_timer_reset(c);
    double *d_Y, *d_X, *d_V, *d_w;
    int rc;
    if ((rc = upload(c, BUF_Y, Y, N, &d_Y))) return rc;
    if ((rc = upload(c, BUF_T, X, N, &d_X))) return rc;
    if ((rc = upload(c, BUF_V, V, N, &d_V))) return rc;
    if ((rc = upload(c, BUF_F, w, Nf, &d_w))) return rc;
    // S accumulates on the device in window order (k_lpv_psd_accum_multi); the parameters never travel to the host
    double* d_S = ws<double>(c, BUF_PSD, (size_t)Nf);
    if (!d_S) return fail(c, LPVS_E_NOMEM, "out of device memory");
    LPVS_CU(c, cudaMemsetAsync(d_S, 0, sizeof(double) * Nf, c->st));
    int any_info = 0;
    for (int64_t k = 0; k < nwin; k++) {
        const int64_t off = k * hop;
        LpvPlan pl;
        if ((rc = lpv_prepare_dev(c, V + off, d_X + off, d_V + off, n, d_w, Nf, Nv, coulomb, normalize, &pl))) return rc;
        int winfo = 0;
        if ((rc = lpv_ls_core(c, pl, d_Y + off, lambda, nullptr, nullptr, fva ? fva + k : nullptr, &winfo, d_S))) {
            if (info) *info = winfo;
            return rc;
        }
        any_info |= winfo;
    }
    if (info) *info = any_info;
    LPVS_CU(c, cudaMemcpyAsync(S, d_S, sizeof(double) * Nf, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    gram_timer_resolve(c);
    return LPVS_OK;
}

int lpvs_ls_spectral_lpv_multi(lpvs_ctx* c, const double* Y, int C, int64_t ldY, const double* X, const double* V,
                               int64_t N, const double* w, int Nf, int Nv, double lambda, int coulomb, int normalize,
                               double* params, double* Sigma0, double* var_e, double* fva, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);  // held across upload + compute: the uploaded channels live in the context's workspace
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (C < 1) return fail(c, LPVS_E_BAD_ARG, "C must be >= 1 (got %d)", C);
    std::vector<int> hinfo((size_t)C, 0);
    int* inf = info ? info : hinfo.data();
    for (int ch = 0; ch < C; ch++) inf[ch] = 0;
    if (!Y || !params) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (ldY < N) return fail(c, LPVS_E_BAD_ARG, "ldY (%lld) must be >= N (%lld)", (long long)ldY, (long long)N);
    gram_timer_reset(c);
    LpvPlan pl;
    int rc = lpv_prepare(c, X, V, N, w, Nf, Nv, coulomb, normalize, &pl);
    if (rc) return rc;
    double* d_Y;
    if ((rc = upload_channels(c, Y, C, ldY, 0, N, &d_Y))) return rc;
    if ((rc = check_channels_finite(c, d_Y, N, N, C))) return rc;
    if ((rc = lpv_ls_core_multi(c, pl, d_Y, N, C, lambda, params, Sigma0, var_e, fva, inf, nullptr))) return rc;
    gram_timer_resolve(c);
    return LPVS_OK;
}

// ls_windowpsd_lpv of C channels: Y, X, V, w go to the device once; per window the tables are built once and every
// channel is solved against them (lpv_ls_core_multi), S[c] accumulating on the device as in lpvs_ls_windowpsd_lpv.
int lpvs_ls_windowpsd_lpv_multi(lpvs_ctx* c, const double* Y, int C, int64_t ldY, const double* X, const double* V,
                                int64_t N, const double* w, int Nf, int Nv, int n, int noverlap, double lambda, int coulomb,
                                int normalize, double* S, double* fva, int64_t* K, int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (K) *K = 0;
    if (C < 1) return fail(c, LPVS_E_BAD_ARG, "C must be >= 1 (got %d)", C);
    if (info)
        for (int ch = 0; ch < C; ch++) info[ch] = 0;
    if (!Y || !X || !V || !w || !S || N <= 0 || Nf <= 0 || Nv <= 0 || n <= 1)
        return fail(c, LPVS_E_BAD_ARG, "bad LPV window arguments");
    if (ldY < N) return fail(c, LPVS_E_BAD_ARG, "ldY (%lld) must be >= N (%lld)", (long long)ldY, (long long)N);
    if (noverlap < 0) noverlap = n >> 1;  // src/windows.jl:97
    if (noverlap >= n) return fail(c, LPVS_E_BAD_ARG, "noverlap must be smaller than the window length");
    const int64_t hop = n - noverlap;
    const int64_t nwin = N >= n ? (N - n) / hop + 1 : 0;
    if (K) *K = nwin;
    for (long long i = 0; i < (long long)Nf * C; i++) S[i] = 0.0;
    if (nwin == 0) return LPVS_OK;
    gram_timer_reset(c);
    double *d_Y, *d_X, *d_V, *d_w;
    int rc;
    if ((rc = upload_channels(c, Y, C, ldY, 0, N, &d_Y))) return rc;
    if ((rc = upload(c, BUF_T, X, N, &d_X))) return rc;
    if ((rc = upload(c, BUF_V, V, N, &d_V))) return rc;
    if ((rc = upload(c, BUF_F, w, Nf, &d_w))) return rc;
    if ((rc = check_channels_finite(c, d_Y, N, N, C))) return rc;
    double* d_S = ws<double>(c, BUF_PSD, (size_t)Nf * C);
    if (!d_S) return fail(c, LPVS_E_NOMEM, "out of device memory");
    LPVS_CU(c, cudaMemsetAsync(d_S, 0, sizeof(double) * Nf * C, c->st));
    std::vector<int> any_info((size_t)C, 0), winfo((size_t)C, 0);
    for (int64_t k = 0; k < nwin; k++) {
        const int64_t off = k * hop;
        LpvPlan pl;
        if ((rc = lpv_prepare_dev(c, V + off, d_X + off, d_V + off, n, d_w, Nf, Nv, coulomb, normalize, &pl))) return rc;
        if ((rc = lpv_ls_core_multi(c, pl, d_Y + off, N, C, lambda, nullptr, nullptr, nullptr, fva ? fva + k * C : nullptr,
                                    winfo.data(), d_S))) {
            if (info)
                for (int ch = 0; ch < C; ch++) info[ch] = winfo[ch];
            if (rc == LPVS_E_NOT_SPD) {
                const std::string msg = c->err;
                return fail(c, rc, "window %lld: %s", (long long)k, msg.c_str());
            }
            return rc;
        }
        for (int ch = 0; ch < C; ch++) any_info[ch] |= winfo[ch];
    }
    if (info)
        for (int ch = 0; ch < C; ch++) info[ch] = any_info[ch];
    LPVS_CU(c, cudaMemcpyAsync(S, d_S, sizeof(double) * Nf * C, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    gram_timer_resolve(c);
    return LPVS_OK;
}

int lpvs_admm_create_fourier(lpvs_ctx* c, const double* y, const double* t, int64_t N, const double* f, int Nf,
                             const double* W, int prox_kind, double prox_param, double mu, const double* x0, int init,
                             double lambda_init, lpvs_admm** out) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (!out) return fail(c, LPVS_E_BAD_ARG, "null handle pointer");
    *out = nullptr;
    if (!y || !t || N <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (!(mu > 0.0) || mu > 1.0) return fail(c, LPVS_E_BAD_ARG, "mu should be in (0, 1]");  // src/lasso.jl:143
    if (prox_kind < LPVS_PROX_L1 || prox_kind > LPVS_PROX_BALL_L0)
        return fail(c, LPVS_E_BAD_ARG, "prox kind %d not valid for the Fourier problem", prox_kind);
    gram_timer_reset(c);
    FourierPlan pl;
    int rc = make_fourier_plan(c, f, Nf, &pl);
    if (rc) return rc;
    if ((rc = admm_check_size(c, pl.Np))) return rc;
    double *d_t, *d_y, *d_W;
    if ((rc = upload(c, BUF_T, t, N, &d_t))) return rc;
    if ((rc = upload(c, BUF_Y, y, N, &d_y))) return rc;
    if ((rc = upload(c, BUF_W, W, N, &d_W))) return rc;
    const long long Np = pl.Np;
    double* d_x0 = nullptr;
    if (init) {
        // fourier_solve(A,y,zerofreq,lambda): unweighted ridge LS with ridge lambda^2 (Q14, src/lasso.jl:92,112)
        double* d_x;
        int inf = 0;
        if ((rc = ls_solve_dev(c, pl, d_t, d_y, nullptr, nullptr, N, 1, lambda_init * lambda_init, c->jitter != 0,
                               &d_x, &inf)))
            return rc;
        d_x0 = ws<double>(c, BUF_X, (size_t)Np);
        if (!d_x0) return fail(c, LPVS_E_NOMEM, "out of device memory");
        LPVS_CU(c, cudaMemcpyAsync(d_x0, d_x, sizeof(double) * Np, cudaMemcpyDeviceToDevice, c->st));
    } else if (x0) {
        double* d_ref;
        if ((rc = upload(c, BUF_MISC, x0, pl.Nreg, &d_ref))) return rc;
        d_x0 = ws<double>(c, BUF_X, (size_t)Np);
        if (!d_x0) return fail(c, LPVS_E_NOMEM, "out of device memory");
        launch_scatter_ref_vec(c, d_ref, pl.Nf, pl.zero_first, pl.Nreg, pl.Np, d_x0);
    }
    double* d_G = nullptr;
    if ((rc = admm_check_memory(c, Np))) return rc;
    if (cudaMalloc(&d_G, sizeof(double) * Np * Np) != cudaSuccess) {
        cudaGetLastError();
        return fail(c, LPVS_E_NOMEM, "out of device memory (Gram %lld MB)", (long long)(Np * Np * 8 >> 20));
    }
    double* d_B = ws<double>(c, BUF_B, (size_t)2 * Np);
    if (!d_B) {
        cudaFree(d_G);
        return fail(c, LPVS_E_NOMEM, "out of device memory");
    }
    if ((rc = gram_single(c, pl, d_t, d_y, nullptr, d_W, N, 1, d_G, d_B))) {
        cudaFree(d_G);
        return rc;
    }
    lpvs_admm* h = admm_new(c);
    admm_set_problem(h, 0, pl.Np, pl.Nf, pl.zero_first, pl.Nreg, pl.Nf, prox_kind, prox_param, mu, W ? 1 : 0, 0, 0);
    if ((rc = admm_finish_create(c, h, d_G, d_B, d_x0)) || (rc = inputs_finite(c))) {
        admm_delete(h);
        return rc;
    }
    gram_timer_resolve(c);
    *out = h;
    return LPVS_OK;
}

int lpvs_admm_create_lpv(lpvs_ctx* c, const double* y, const double* X, const double* V, int64_t N, const double* w,
                         int Nf, int Nv, int coulomb, int normalize, double lambda, double mu, lpvs_admm** out) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (!out) return fail(c, LPVS_E_BAD_ARG, "null handle pointer");
    *out = nullptr;
    if (!y) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    if (!(mu > 0.0) || mu > 1.0) return fail(c, LPVS_E_BAD_ARG, "mu should be in (0, 1]");
    gram_timer_reset(c);
    LpvPlan pl;
    int rc = lpv_prepare(c, X, V, N, w, Nf, Nv, coulomb, normalize, &pl);
    if (rc) return rc;
    if ((rc = admm_check_size(c, pl.Np))) return rc;
    double* d_y;
    if ((rc = upload(c, BUF_Y, y, N, &d_y))) return rc;
    const long long Np = pl.Np;
    double* d_G = nullptr;
    if ((rc = admm_check_memory(c, Np))) return rc;
    if (cudaMalloc(&d_G, sizeof(double) * Np * Np) != cudaSuccess) {
        cudaGetLastError();
        return fail(c, LPVS_E_NOMEM, "out of device memory (Gram %lld MB)", (long long)(Np * Np * 8 >> 20));
    }
    double* d_B = ws<double>(c, BUF_B, (size_t)2 * Np);
    if (!d_B) {
        cudaFree(d_G);
        return fail(c, LPVS_E_NOMEM, "out of device memory");
    }
    if ((rc = lpv_gram(c, pl, d_y, d_G, d_B))) {
        cudaFree(d_G);
        return rc;
    }
    // groups (src/lasso.jl:47-55): permuted position p = f*(len/Nf) + kk  <->  un-permuted f + kk*Nf; group g covers
    // permuted positions [g*2Nv, (g+1)*2Nv), g < Nf.  With coulomb the groups cover only the first half (Q16).
    const int ncc = pl.ncc, len = 2 * ncc, per_f = len / Nf;
    std::vector<int> goff((size_t)Nf + 2), gmem;
    std::vector<char> covered((size_t)Np, 0);
    gmem.reserve((size_t)Np);
    for (int g = 0; g < Nf; g++) {
        goff[g] = (int)gmem.size();
        for (int p = g * 2 * Nv; p < (g + 1) * 2 * Nv && p < len; p++) {
            int fq = p / per_f, kk = p % per_f;
            int j = fq + kk * Nf;
            int cc = j < ncc ? j : j - ncc, part = j < ncc ? 0 : 1;
            int idx = (cc >> 6) * 128 + part * 64 + (cc & 63);
            gmem.push_back(idx);
            covered[idx] = 1;
        }
    }
    goff[Nf] = (int)gmem.size();
    for (int i = 0; i < Np; i++)
        if (!covered[i]) gmem.push_back(i);
    goff[Nf + 1] = (int)gmem.size();
    lpvs_admm* h = admm_new(c);
    admm_set_problem(h, 1, pl.Np, ncc, 0, len, ncc, LPVS_PROX_GROUP_L2, lambda, mu, 0, Nf, pl.Nvv);
    if ((rc = admm_set_groups(c, h, goff, gmem)) || (rc = admm_finish_create(c, h, d_G, d_B, nullptr)) ||
        (rc = inputs_finite(c))) {
        admm_delete(h);
        const int rcf = inputs_finite(c);  // a NaN basis breaks the factorisation first: report the cause
        return rcf ? rcf : rc;
    }
    gram_timer_resolve(c);
    *out = h;
    return LPVS_OK;
}

int lpvs_ls_sparse_spectral(lpvs_ctx* c, const double* y, const double* t, int64_t N, const double* f, int Nf,
                            const double* W, int prox_kind, double prox_param, double mu, int init, double lambda_init,
                            int64_t iters, double tol, double* x, int64_t* iters_done, double* residual) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);  // create / run / result / free as one serialised unit
    lpvs_admm* h = nullptr;
    int rc = lpvs_admm_create_fourier(c, y, t, N, f, Nf, W, prox_kind, prox_param, mu, nullptr, init, lambda_init, &h);
    if (rc) return rc;
    int conv = 0;
    rc = lpvs_admm_run(h, iters, tol, iters_done, residual, &conv);
    if (!rc) rc = lpvs_admm_result(h, x);
    lpvs_admm_free(h);
    return rc;
}

int lpvs_ls_sparse_spectral_lpv(lpvs_ctx* c, const double* y, const double* X, const double* V, int64_t N,
                                const double* w, int Nf, int Nv, int coulomb, int normalize, double lambda, double mu,
                                int64_t iters, double tol, double* params, int64_t* iters_done, double* residual) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);  // create / run / result / free as one serialised unit
    lpvs_admm* h = nullptr;
    int rc = lpvs_admm_create_lpv(c, y, X, V, N, w, Nf, Nv, coulomb, normalize, lambda, mu, &h);
    if (rc) return rc;
    int conv = 0;
    rc = lpvs_admm_run(h, iters, tol, iters_done, residual, &conv);
    if (!rc) rc = lpvs_admm_result(h, params);
    lpvs_admm_free(h);
    return rc;
}

// ---- row-sharded Gram (SURVEY 8e): partial G,b on device; the host all-reduces d_packed across ranks ----
int64_t lpvs_packed_size(int Nf) {
    long long nb = (Nf + FB - 1) / FB;
    long long Np = nb * TB;
    return Np * Np + 2 * Np;
}

int lpvs_gram_partial_dev(lpvs_ctx* c, const double* d_y, const double* d_u, const double* d_t, const double* d_W,
                          int64_t N, const double* f, int Nf, double* d_packed) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (!d_t || !d_packed || N <= 0) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    gram_timer_reset(c);
    FourierPlan pl;
    int rc = make_fourier_plan(c, f, Nf, &pl);
    if (rc) return rc;
    const long long Np = pl.Np;
    LPVS_CU(c, cudaMemsetAsync(d_packed + Np * Np, 0, sizeof(double) * 2 * Np, c->st));
    int nrhs = d_y ? (d_u ? 2 : 1) : 0;
    if ((rc = gram_single(c, pl, d_t, d_y, d_u, d_W, N, nrhs, d_packed, d_packed + Np * Np))) return rc;
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    gram_timer_resolve(c);
    return LPVS_OK;
}

int lpvs_solve_packed_dev(lpvs_ctx* c, double* d_packed, const double* f, int Nf, int nrhs, double ridge, double* x,
                          int* info) {
    if (!c) return LPVS_E_BAD_ARG;
    Lock lk(c->mu);
    CallTimer call_timer(c);
    cudaSetDevice(c->device);
    if (info) *info = 0;
    if (!d_packed || !x || nrhs < 1 || nrhs > 2) return fail(c, LPVS_E_BAD_ARG, "bad arguments");
    FourierPlan pl;
    int rc = make_fourier_plan(c, f, Nf, &pl);
    if (rc) return rc;
    const long long Np = pl.Np;
    int pinfo = 0;
    // same policy as the single-GPU weighted ls_spectral: on breakdown re-factor once with the jitter ridge
    double* d_keep = c->jitter ? ws<double>(c, BUF_YINV, (size_t)Np * Np + 2 * Np) : nullptr;
    if (d_keep)
        LPVS_CU(c, cudaMemcpyAsync(d_keep, d_packed, sizeof(double) * (Np * Np + 2 * Np), cudaMemcpyDeviceToDevice, c->st));
    double maxdiag = 0.0;
    if (d_keep) {
        double* d_md = ws<double>(c, BUF_SUMS, 8);
        if (!d_md) return fail(c, LPVS_E_NOMEM, "out of device memory");
        launch_max_diag(d_packed, Np * Np, pl.Np, pl.Nf, pl.zero_first, d_md, 1, c->st);
        c->launches++;
        LPVS_CU(c, cudaMemcpyAsync(&maxdiag, d_md, sizeof(double), cudaMemcpyDeviceToHost, c->st));
    }
    if ((rc = factor_solve(c, pl.Nf, pl.zero_first, pl.Np, d_packed, d_packed + Np * Np, nrhs, ridge, 1, &pinfo)))
        return rc;
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    if (pinfo && d_keep) {
        LPVS_CU(c, cudaMemcpyAsync(d_packed, d_keep, sizeof(double) * (Np * Np + 2 * Np), cudaMemcpyDeviceToDevice, c->st));
        const double jr = std::max(ridge, (double)pl.Nreg * 2.220446049250313e-16 * maxdiag);
        if ((rc = factor_solve(c, pl.Nf, pl.zero_first, pl.Np, d_packed, d_packed + Np * Np, nrhs, jr, 1, &pinfo)))
            return rc;
        LPVS_CU(c, cudaStreamSynchronize(c->st));
        if (!pinfo && info) *info = LPVS_INFO_JITTER;
    }
    if (pinfo) {
        if (info) *info = pinfo;
        return fail(c, LPVS_E_NOT_SPD, "Cholesky breakdown at internal pivot %d", pinfo);
    }
    double* d_out = ws<double>(c, BUF_X, (size_t)2 * nrhs * Nf);
    if (!d_out) return fail(c, LPVS_E_NOMEM, "out of device memory");
    launch_x_to_complex(c, d_packed + Np * Np, pl.Np, Nf, pl.zero_first, nrhs, d_out);
    LPVS_CU(c, cudaMemcpyAsync(x, d_out, sizeof(double) * 2 * nrhs * Nf, cudaMemcpyDeviceToHost, c->st));
    LPVS_CU(c, cudaStreamSynchronize(c->st));
    return LPVS_OK;
}

}  // extern "C"
