"""GPU: ls_spectral_lpv / ls_windowpsd_lpv of C output channels sharing X and V (lpvs_ls_spectral_lpv_multi,
lpvs_ls_windowpsd_lpv_multi) against the oracle, the single-channel calls, and their exact properties.

Every channel is scaled by 10^((c mod 7) - 3) and judged against its own norm, so a quiet channel cannot hide behind a loud
one.  Bars as tests/test_gpu_rankdef.py::test_lpv_default_lambda: max(1e-9, 50 cond([Ar; lam I]) eps) for the parameters
(against the literal gelsy solve and the QR solve of [Ar; lam I]), 1e-9 for fva, 1e-4 for Sigma.  Sigma is the inverse of
Ar'Ar + lam I, whose condition number at lam = 1e-8 bounds its accuracy; the coulomb and unnormalised parity cases use
Nv = 6, as that test's coulomb case does, where the 1e-4 bar holds for the single-channel call too.  A channel can take a
different route from its single call where its first refinement step lands on the 0.05 contraction threshold (as stated for
ls_spectral_multi); both answers meet the bar, so the comparison with single calls checks the values to the bar and the
routes only on channels that are far from that threshold."""
import ctypes as C
import warnings

import numpy as np
import pytest
import scipy.linalg as sla

from oracle import lpvs_oracle as o

pytestmark = pytest.mark.gpu

EPS = np.finfo(float).eps
C_TOL = 50.0


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(b)


def scale(c):
    return 10.0 ** ((c % 7) - 3)


def cond_aug(A, lam):
    s = np.linalg.svd(A, compute_uv=False)
    smin = s[-1] if A.shape[0] >= A.shape[1] else 0.0
    return np.hypot(s[0], lam) / np.hypot(smin, lam)


def problem(N, nch, seed=0, coulomb=False):
    """X, V of an LPV record; channel c: the record's output, white noise or a V-modulated sinusoid, scaled."""
    Y0, V, X = o.generate_lpv_signal(N, seed=seed)
    if coulomb:
        V = V - 0.5 + 1e-3
    rng = np.random.default_rng(seed + 100)
    Y = np.empty((N, nch))
    for c in range(nch):
        k = c % 3
        if k == 0:
            y = Y0 + 0.01 * rng.standard_normal(N)
        elif k == 1:
            y = rng.standard_normal(N)
        else:
            y = np.sin(2 * np.pi * (1 + c % 5) * X) * (1 + V) + 0.1 * rng.standard_normal(N)
        Y[:, c] = scale(c) * y
    return Y, X, V


def wgrid(Nf):
    return 2 * np.pi * np.arange(1, Nf + 1, dtype=float)


def quiet(fn, *a, **k):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return fn(*a, **k)


def multi_abi(ctx, Y, X, V, w, Nv, lam=1e-8, coulomb=False, normalize=True, ldY=None, want_sigma=True):
    """lpvs_ls_spectral_lpv_multi on Y (N x C) with leading dimension ldY -> (params (C, ncc), Sigma0, var_e, fva, info)."""
    N, nch = Y.shape
    ldY = ldY or N
    Yc = np.zeros((nch, ldY))
    Yc[:, :N] = Y.T
    ncc = len(w) * (2 if coulomb else 1) * Nv
    params = np.empty((nch, ncc), dtype=np.complex128)
    S0 = np.empty((2 * ncc, 2 * ncc)) if want_sigma else None
    ve, fva, info = np.empty(nch), np.empty(nch), np.zeros(nch, dtype=np.int32)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    ctx.check(ctx.lib.lpvs_ls_spectral_lpv_multi(ctx.h, p(Yc), nch, ldY, p(np.ascontiguousarray(X)),
                                                 p(np.ascontiguousarray(V)), N, p(np.ascontiguousarray(w)), len(w), Nv,
                                                 lam, int(coulomb), int(normalize), p(params), p(S0), p(ve), p(fva),
                                                 info.ctypes.data_as(C.POINTER(C.c_int))))
    return params, S0, ve, fva, info


def single_abi(ctx, y, X, V, w, Nv, lam=1e-8, coulomb=False, normalize=True):
    """lpvs_ls_spectral_lpv -> (params, Sigma, fva, info)."""
    ncc = len(w) * (2 if coulomb else 1) * Nv
    params = np.empty(ncc, dtype=np.complex128)
    Sig = np.empty((2 * ncc, 2 * ncc))
    fva, info = C.c_double(0.0), C.c_int(0)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    ctx.check(ctx.lib.lpvs_ls_spectral_lpv(ctx.h, p(np.ascontiguousarray(y)), p(np.ascontiguousarray(X)),
                                           p(np.ascontiguousarray(V)), len(y), p(np.ascontiguousarray(w)), len(w), Nv, lam,
                                           int(coulomb), int(normalize), p(params), p(Sig), C.byref(fva), C.byref(info)))
    return params, Sig, fva.value, info.value


# ---- parity against the oracle -----------------------------------------------------------------------------------------


@pytest.mark.parametrize("lam,Nv,coulomb,normalize", [(1e-8, 10, False, True), (1e-8, 50, False, True),
                                                      (1e-8, 6, True, True), (1e-8, 6, False, False),
                                                      (0.02, 10, False, True), (0.02, 50, True, False)])
def test_parity_with_oracle(ctx, lam, Nv, coulomb, normalize):
    import lpvspectral_jl_b200 as lp

    N, nch, Nf = 500, 5, 10
    Y, X, V = problem(N, nch, coulomb=coulomb)
    w = wgrid(Nf)
    out, info = quiet(lp.ls_spectral_lpv_multi, Y, X, V, w, Nv, λ=lam, coulomb=coulomb, normalize=normalize, ctx=ctx,
                      return_info=True)
    Ar = o.lpv_regressor(X, V, w, Nv, normalize, coulomb)
    n2 = Ar.shape[1]
    tol = max(1e-9, C_TOL * cond_aug(Ar, lam) * EPS)
    M = np.vstack([Ar, lam * np.eye(n2)])
    Q, R = np.linalg.qr(M)
    XQ = sla.solve_triangular(R, Q[:N].T @ Y, check_finite=False)
    for c in range(nch):
        sr = o.ls_spectral_lpv(Y[:, c], X, V, w, Nv, lam=lam, coulomb=coulomb, normalize=normalize, mode="literal")
        xq = XQ[: n2 // 2, c] + 1j * XQ[n2 // 2:, c]
        se = out[c]
        print(f"lam={lam} Nv={Nv} c={c} info={info[c]}: gelsy {rel(se.x, sr.x):.2e} qr {rel(se.x, xq):.2e} tol {tol:.2e}")
        assert rel(se.x, sr.x) <= tol and rel(se.x, xq) <= tol
        assert abs(se.fva - sr.fva) <= 1e-9
        assert rel(se.Σ, sr.Sigma) <= 1e-4
        _, Ss, _, _ = single_abi(ctx, Y[:, c], X, V, w, Nv, lam=lam, coulomb=coulomb, normalize=normalize)
        assert rel(se.Σ, Ss) <= 1e-6  # the same inverse as the single call's, scaled by its own var(e)


# ---- against the single-channel call -----------------------------------------------------------------------------------


@pytest.mark.parametrize("lam,Nv", [(1e-8, 10), (0.02, 20)])
def test_matches_single_calls(ctx, lam, Nv):
    N, nch, Nf = 600, 6, 8
    Y, X, V = problem(N, nch, seed=3)
    w = wgrid(Nf)
    params, S0, ve, fva, info = multi_abi(ctx, Y, X, V, w, Nv, lam=lam)
    tol = max(1e-9, C_TOL * cond_aug(o.lpv_regressor(X, V, w, Nv), lam) * EPS)
    for c in range(nch):
        xs, Ss, fs, inf = single_abi(ctx, Y[:, c], X, V, w, Nv, lam=lam)
        assert rel(params[c], xs) <= tol
        assert abs(fva[c] - fs) <= 1e-9
        assert rel(ve[c] * S0, Ss) <= 1e-4
        assert info[c] == inf, (c, info, inf)


def test_sinusoid_noise_and_zero_channels_take_their_single_routes(ctx):
    N, Nf, Nv = 400, 6, 10
    Y0, X, V = problem(N, 2, seed=5)
    Y = np.stack([Y0[:, 0], Y0[:, 1], np.zeros(N)], axis=1)
    w = wgrid(Nf)
    for lam in (1e-8, 0.02):
        params, _, _, fva, info = multi_abi(ctx, Y, X, V, w, Nv, lam=lam)
        singles = [single_abi(ctx, Y[:, c], X, V, w, Nv, lam=lam) for c in range(3)]
        print(f"lam={lam}: multi routes {list(info)}, single routes {[s[3] for s in singles]}")
        assert [int(i) for i in info] == [s[3] for s in singles]
        assert np.all(params[2] == 0)
        tol = max(1e-9, C_TOL * cond_aug(o.lpv_regressor(X, V, w, Nv), lam) * EPS)
        for c in range(2):
            assert rel(params[c], singles[c][0]) <= tol


# ---- exact properties --------------------------------------------------------------------------------------------------


def test_channel_independence_is_bitwise(ctx):
    N, nch, Nf, Nv = 500, 17, 8, 10
    Y, X, V = problem(N, nch, seed=7)
    w = wgrid(Nf)
    ref = multi_abi(ctx, Y, X, V, w, Nv)
    perm = np.random.default_rng(0).permutation(nch)
    got = multi_abi(ctx, Y[:, perm], X, V, w, Nv)
    for k in (0, 2, 3, 4):  # params, var_e, fva, info
        assert np.array_equal(got[k], ref[k][perm], equal_nan=True)
    assert np.array_equal(got[1], ref[1])  # Sigma0 does not depend on Y
    sub = [3, 11, 16]
    got = multi_abi(ctx, Y[:, sub], X, V, w, Nv)
    for k in (0, 2, 3, 4):
        assert np.array_equal(got[k], ref[k][sub], equal_nan=True)
    for c in (0, 9, 16):  # C = 1
        got = multi_abi(ctx, Y[:, [c]], X, V, w, Nv)
        for k in (0, 2, 3, 4):
            assert np.array_equal(got[k][0], ref[k][c], equal_nan=True)
    dup = [5, 5, 2, 5]
    got = multi_abi(ctx, Y[:, dup], X, V, w, Nv)
    for k in (0, 2, 3, 4):
        assert np.array_equal(got[k], ref[k][dup], equal_nan=True)


# ---- edges: chunk widths, 64-column blocks, padded ldY, the dual route ---------------------------------------------------


@pytest.mark.parametrize("nch", [1, 3, 4, 5, 16, 17, 32, 33])
def test_channel_counts(ctx, nch):
    N, Nf, Nv = 300, 8, 8  # ncc = 64
    Y, X, V = problem(N, nch, seed=nch)
    w = wgrid(Nf)
    params, S0, ve, fva, info = multi_abi(ctx, Y, X, V, w, Nv, ldY=N + 3 if nch % 2 else None)
    tol = max(1e-9, C_TOL * cond_aug(o.lpv_regressor(X, V, w, Nv), 1e-8) * EPS)
    for c in range(nch):
        xs, _, fs, _ = single_abi(ctx, Y[:, c], X, V, w, Nv)
        assert rel(params[c], xs) <= tol, c
        assert abs(fva[c] - fs) <= 1e-9


@pytest.mark.parametrize("Nf,Nv,lam", [(7, 9, 1e-8), (8, 8, 1e-8), (5, 13, 1e-8), (13, 10, 0.02)])
def test_block_edges_against_oracle(ctx, Nf, Nv, lam):
    N, nch = 400, 4  # ncc = 63, 64, 65, 130
    Y, X, V = problem(N, nch, seed=Nf)
    w = wgrid(Nf)
    params, S0, ve, fva, info = multi_abi(ctx, Y, X, V, w, Nv, lam=lam, ldY=N + 64)
    Ar = o.lpv_regressor(X, V, w, Nv)
    tol = max(1e-9, C_TOL * cond_aug(Ar, lam) * EPS)
    for c in range(nch):
        sr = o.ls_spectral_lpv(Y[:, c], X, V, w, Nv, lam=lam)
        assert rel(params[c], sr.x) <= tol
        assert abs(fva[c] - sr.fva) <= 1e-9
        assert rel(ve[c] * S0, sr.Sigma) <= 1e-4


@pytest.mark.parametrize("lam", [1e-8, 0.02])
def test_more_unknowns_than_samples(ctx, lam):
    """2 ncc >= N: the sample-space (dual) route, shared by the channels."""
    N, nch, Nf, Nv = 100, 5, 8, 8
    Y, X, V = problem(N, nch, seed=11)
    w = wgrid(Nf)
    params, S0, ve, fva, info = multi_abi(ctx, Y, X, V, w, Nv, lam=lam)
    tol = max(1e-9, C_TOL * cond_aug(o.lpv_regressor(X, V, w, Nv), lam) * EPS)
    print(f"lam={lam}: routes {list(info)}")
    for c in range(nch):
        sr = o.ls_spectral_lpv(Y[:, c], X, V, w, Nv, lam=lam)
        xs, _, _, inf = single_abi(ctx, Y[:, c], X, V, w, Nv, lam=lam)
        assert rel(params[c], sr.x) <= tol and rel(params[c], xs) <= tol
        assert info[c] == inf


# ---- windowed ----------------------------------------------------------------------------------------------------------


def windowed_abi(ctx, Y, X, V, w, Nv, nw, noverlap, multi=True):
    N, nch = Y.shape
    n = N // nw
    Kw = int(ctx.lib.lpvs_window_count(N, n, noverlap))
    K = C.c_int64(0)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    Xc, Vc, wc = np.ascontiguousarray(X), np.ascontiguousarray(V), np.ascontiguousarray(w)
    if multi:
        S, fva, info = np.empty((nch, len(w))), np.empty((Kw, nch)), np.zeros(nch, dtype=np.int32)
        ctx.check(ctx.lib.lpvs_ls_windowpsd_lpv_multi(ctx.h, p(np.ascontiguousarray(Y.T)), nch, N, p(Xc), p(Vc), N, p(wc),
                                                      len(w), Nv, n, noverlap, 1e-8, 0, 1, p(S), p(fva), C.byref(K),
                                                      info.ctypes.data_as(C.POINTER(C.c_int))))
        assert K.value == Kw
        return S, fva, info
    S, fva, info = np.empty(len(w)), np.empty(Kw), C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_windowpsd_lpv(ctx.h, p(np.ascontiguousarray(Y)), p(Xc), p(Vc), N, p(wc), len(w), Nv, n,
                                            noverlap, 1e-8, 0, 1, p(S), p(fva), C.byref(K), C.byref(info)))
    return S, fva, info.value


@pytest.mark.parametrize("nw,noverlap", [(10, 0), (5, 100)])
def test_windowed_against_single_and_oracle(ctx, nw, noverlap):
    import lpvspectral_jl_b200 as lp

    N, nch, Nf, Nv = 2000, 5, 8, 12
    Y, X, V = problem(N, nch, seed=1)
    w = wgrid(Nf)
    S = quiet(lp.ls_windowpsd_lpv_multi, Y, X, V, w, Nv, nw, noverlap, ctx=ctx)
    assert S.shape == (Nf, nch)
    Sm, fvam, infom = windowed_abi(ctx, Y, X, V, w, Nv, nw, noverlap)
    assert np.array_equal(Sm.T, S)
    for c in range(nch):
        Ss, fvas, infos = windowed_abi(ctx, Y[:, [c]], X, V, w, Nv, nw, noverlap, multi=False)
        Sr = o.ls_windowpsd_lpv(Y[:, c], X, V, w, Nv, nw, noverlap)
        print(f"nw={nw} noverlap={noverlap} c={c}: vs single {rel(S[:, c], Ss):.2e} vs oracle {rel(S[:, c], Sr):.2e}")
        assert rel(S[:, c], Ss) <= 1e-6 and rel(S[:, c], Sr) <= 1e-4
        assert np.max(np.abs(fvam[:, c] - fvas)) <= 1e-9
        assert infom[c] == infos


# ---- errors ------------------------------------------------------------------------------------------------------------


def test_errors(ctx):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    N, nch, Nf, Nv = 300, 5, 6, 8
    Y, X, V = problem(N, nch, seed=2)
    w = wgrid(Nf)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    Yc = np.ascontiguousarray(Y.T)
    params = np.empty(nch * Nf * Nv, dtype=np.complex128)
    info = np.zeros(nch, dtype=np.int32)
    ip = info.ctypes.data_as(C.POINTER(C.c_int))
    args = (p(X), p(V), N, p(w), Nf, Nv, 1e-8, 0, 1, p(params), None, None, None, ip)
    assert ctx.lib.lpvs_ls_spectral_lpv_multi(ctx.h, p(Yc), 0, N, *args) == L.E_BAD_ARG
    assert ctx.lib.lpvs_ls_spectral_lpv_multi(ctx.h, p(Yc), nch, N - 1, *args) == L.E_BAD_ARG
    assert ctx.lib.lpvs_ls_spectral_lpv_multi(ctx.h, None, nch, N, *args) == L.E_BAD_ARG
    S, K = np.empty((nch, Nf)), C.c_int64(0)
    wargs = (p(X), p(V), N, p(w), Nf, Nv, N // 3, 0, 1e-8, 0, 1, p(S), None, C.byref(K), ip)
    assert ctx.lib.lpvs_ls_windowpsd_lpv_multi(ctx.h, p(Yc), 0, N, *wargs) == L.E_BAD_ARG
    assert ctx.lib.lpvs_ls_windowpsd_lpv_multi(ctx.h, p(Yc), nch, N - 1, *wargs) == L.E_BAD_ARG
    Yn = Y.copy()
    Yn[17, 3] = np.nan
    Yn[40, 4] = np.inf
    for fn in (lp.ls_spectral_lpv_multi, lp.ls_windowpsd_lpv_multi):
        with pytest.raises(L.LpvsError, match="channel 3"):
            quiet(fn, Yn, X, V, w, Nv, ctx=ctx)
        with pytest.raises(ValueError, match="degenerate"):  # LPVS_E_BAD_ARG
            quiet(fn, Y, X, np.full(N, 0.5), w, Nv, ctx=ctx)
    # LPVS_OPT_JITTER = 0: one plain Cholesky with ridge lam^2; more unknowns than samples breaks it down
    Nvb = 40
    ctx.set_option(L.OPT_JITTER, 0)
    try:
        with pytest.raises(L.NotPositiveDefinite):
            quiet(lp.ls_spectral_lpv, Y[:, 0], X, V, w, Nvb, ctx=ctx)
        info2 = np.zeros(nch, dtype=np.int32)
        params2 = np.empty(nch * Nf * Nvb, dtype=np.complex128)
        rc = ctx.lib.lpvs_ls_spectral_lpv_multi(ctx.h, p(Yc), nch, N, p(X), p(V), N, p(w), Nf, Nvb, 1e-8, 0, 1,
                                                p(params2), None, None, None, info2.ctypes.data_as(C.POINTER(C.c_int)))
        assert rc == L.E_NOT_SPD and info2[0] > 0 and np.all(info2 == info2[0])
        with pytest.raises(L.NotPositiveDefinite, match="window 0"):
            quiet(lp.ls_windowpsd_lpv_multi, Y, X, V, w, Nvb, 2, ctx=ctx)
    finally:
        ctx.set_option(L.OPT_JITTER, 1)
