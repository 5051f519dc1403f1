"""GPU: cross-spectral / coherence matrices of C channels from one factorisation per window (lpvs_ls_window_matrix_sums).

Entry (i, j) must match the two-channel estimators on channels i and j, the PSD column c ls_windowpsd(Y[:, c]), to
max(1e-12, 40 cond eps) relative (cond = the largest cond(A'WA + lam I) over the windows): both sides solve the same normal
equations with different kernels.  -m gpu."""
import ctypes as C

import numpy as np
import pytest

from oracle import lpvs_oracle as o

import oracle_matrix as om

pytestmark = pytest.mark.gpu

EPS = 2.220446049250313e-16


@pytest.fixture(params=[0, 1, 2, 3], ids=["auto", "chain", "direct", "chain_ref"])
def phase(ctx, request):
    from lpvspectral_jl_b200 import _lib as L

    ctx.set_option(L.OPT_PHASE_MODE, request.param)
    try:
        yield request.param
    finally:
        ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_AUTO)


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(b)


def record(N, C, seed, T=10.0):
    rng = np.random.default_rng(seed)
    t = np.sort(T * rng.random(N))
    common = np.sin(2 * np.pi * 7.3 * t)
    Y = np.stack([(0.3 + 0.1 * c) * common + np.cos(2 * np.pi * (2.1 + 0.37 * c) * t + c)
                  + 0.4 * rng.standard_normal(N) for c in range(C)], axis=1)
    return t, Y


def max_cond(t, f, n, noverlap, W, lam=1e-10):
    hop = n - noverlap
    K = o.arraysplit_count(len(t), n, noverlap)
    worst = 1.0
    for k in range(K):
        A, _ = o.get_fourier_regressor(t[k * hop:k * hop + n], f)
        worst = max(worst, np.linalg.cond((A.T * W) @ A + lam * np.eye(A.shape[1])))
    return worst


def bar(cond):
    return max(1e-12, 40.0 * cond * EPS)


# (N, C, nw, f) -- irregular t throughout; uniform grids with f0 = 0 and f0 != 0, a non-uniform grid (DIRECT), Nf = 1 / 65 / 300
CASES = {
    "c3_nf65_f0zero": (2400, 3, 6, lambda T: np.arange(65) * 2.0 / T),
    "c17_nf300_f0": (7200, 17, 4, lambda T: (np.arange(300) + 3) * 2.0 / T),
    "c64_nf1": (2000, 64, 5, lambda T: np.array([3.5 / T])),
    "c2_nf65_nonuniform": (2400, 2, 6, lambda T: np.cumsum(1.5 + np.random.default_rng(2).random(65)) / T),
    "c1_nf65": (2400, 1, 6, lambda T: np.arange(65) * 2.0 / T),
}


@pytest.mark.parametrize("case", list(CASES))
def test_matrix_matches_pairwise_estimators(ctx, phase, case):
    import lpvspectral_jl_b200 as lp

    N, nch, nw, fgen = CASES[case]
    if case.endswith("nonuniform") and phase in (1, 3):
        pytest.skip("the chain modes need a uniform grid")
    t, Y = record(N, nch, seed=N + nch)
    n = N // nw
    f = fgen(t[n] - t[0])
    S, fr = lp.ls_windowcsd_matrix(Y, t, f, nw=nw, window_func=lp.hanning, ctx=ctx)
    Co, _ = lp.ls_cohere_matrix(Y, t, f, nw=nw, ctx=ctx)
    P, _ = lp.ls_windowpsd_multi(Y, t, f, nw=nw, window_func=lp.hanning, ctx=ctx)
    assert S.shape == (len(f), nch, nch) and Co.shape == S.shape and P.shape == (len(f), nch) and fr is f
    tol = bar(max_cond(t, f, n, n >> 1, o.hanning(n)))
    rng = np.random.default_rng(0)
    pairs = {(0, nch - 1), (nch - 1, 0), (0, 0), (nch // 2, nch // 3)}
    if nch <= 3:
        pairs |= {(i, j) for i in range(nch) for j in range(nch)}
    else:
        pairs |= {tuple(rng.integers(0, nch, 2)) for _ in range(4)}
    for i, j in sorted(pairs):
        Sr, _ = lp.ls_windowcsd(Y[:, i], Y[:, j], t, f, nw=nw, window_func=lp.hanning, ctx=ctx)
        Cr, _ = lp.ls_cohere(Y[:, i], Y[:, j], t, f, nw=nw, ctx=ctx)
        assert rel(S[:, i, j], Sr) <= tol, (i, j, rel(S[:, i, j], Sr), tol)
        assert rel(Co[:, i, j], Cr) <= tol, (i, j, rel(Co[:, i, j], Cr), tol)
    for c in sorted({0, nch - 1, nch // 2}):
        Pr, _ = lp.ls_windowpsd(Y[:, c], t, f, nw=nw, window_func=lp.hanning, ctx=ctx)
        assert rel(P[:, c], Pr) <= tol


@pytest.mark.parametrize("mode", [4, 5], ids=["structured", "structured_ref"])
def test_structured_modes_match_default(ctx, mode):
    import lpvspectral_jl_b200 as lp

    t, Y = record(4800, 5, seed=3)
    nw = 6
    n = 4800 // nw
    f = (np.arange(150) + 1) * 2.0 / (t[n] - t[0])
    S0, _ = lp.ls_windowcsd_matrix(Y, t, f, nw=nw, window_func=lp.hanning, ctx=ctx)
    C0, _ = lp.ls_cohere_matrix(Y, t, f, nw=nw, ctx=ctx)
    with ctx.phase_mode(mode):
        S, _ = lp.ls_windowcsd_matrix(Y, t, f, nw=nw, window_func=lp.hanning, ctx=ctx)
        Co, _ = lp.ls_cohere_matrix(Y, t, f, nw=nw, ctx=ctx)
    # the bars of tests/test_gpu_structured.py: 1e-9 against the default mode
    assert rel(S, S0) <= 1e-9 and rel(Co, C0) <= 1e-9


def test_against_literal_oracle(ctx):
    import lpvspectral_jl_b200 as lp

    t, Y = record(2400, 3, seed=11)
    nw = 6
    n = 400
    f = np.arange(40) * 2.0 / (t[n] - t[0])
    tol = bar(max_cond(t, f, n, n >> 1, o.hanning(n)))
    S, _ = lp.ls_windowcsd_matrix(Y, t, f, nw=nw, window_func=lp.hanning, ctx=ctx)
    Sr, _ = om.ls_windowcsd_matrix(Y, t, f, nw=nw, window_func=o.hanning)
    Co, _ = lp.ls_cohere_matrix(Y, t, f, nw=nw, ctx=ctx)
    Cr, _ = om.ls_cohere_matrix(Y, t, f, nw=nw)
    P, _ = lp.ls_windowpsd_multi(Y, t, f, nw=nw, window_func=lp.hanning, ctx=ctx)
    Pr, _ = om.ls_windowpsd_multi(Y, t, f, nw=nw, window_func=o.hanning)
    for i in range(3):
        assert rel(P[:, i], Pr[:, i]) <= tol
        for j in range(3):
            assert rel(S[:, i, j], Sr[:, i, j]) <= tol and rel(Co[:, i, j], Cr[:, i, j]) <= tol


def _dev_sums(ctx, Y, t, f, W, n, noverlap, lam, k0, k1, ldY=None):
    """lpvs_ls_window_matrix_sums_dev on device copies of Y (channel c at c ldY, ldY >= N) and t."""
    import torch

    dev = torch.device("cuda", ctx.device)
    N, nch = Y.shape
    ldY = N if ldY is None else ldY
    Yp = np.zeros((nch, ldY))
    Yp[:, :N] = Y.T
    Yd = torch.from_numpy(Yp).to(dev)
    td = torch.from_numpy(t).to(dev)
    torch.cuda.synchronize(dev)
    sums = np.zeros((len(f), nch, nch), dtype=np.complex128)
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_window_matrix_sums_dev(ctx.h, C.c_void_p(Yd.data_ptr()), nch, ldY, C.c_void_p(td.data_ptr()), N,
                                                     f.ctypes.data_as(C.c_void_p), len(f), W.ctypes.data_as(C.c_void_p), n,
                                                     noverlap, lam, k0, k1, sums.ctypes.data_as(C.c_void_p),
                                                     C.byref(info)))
    return sums


def test_exact_properties(ctx):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    N, nch, n = 8000, 5, 500
    t, Y = record(N, nch, seed=5)
    f = np.arange(65) * 2.0 / (t[n] - t[0])
    W = o.hanning(n)
    nov = n >> 1
    K = lp.window_count(N, n, nov)
    full = lp.window_matrix_sums(Y, t, f, W, n, nov, 1e-10, 0, K, ctx=ctx)
    # Hermitian bit for bit, real diagonal
    assert np.array_equal(full, np.conj(np.transpose(full, (0, 2, 1))))
    assert np.all(np.einsum("fii->fi", full).imag == 0)
    # several factorisation batches give the same bits
    ctx.set_option(L.OPT_WINDOW_BATCH, 5)
    try:
        small = lp.window_matrix_sums(Y, t, f, W, n, nov, 1e-10, 0, K, ctx=ctx)
    finally:
        ctx.set_option(L.OPT_WINDOW_BATCH, 0)
    assert np.array_equal(small, full)
    # the device-pointer form, and a host matrix with a leading dimension beyond N
    assert np.array_equal(_dev_sums(ctx, Y, t, f, W, n, nov, 1e-10, 0, K), full)
    Yp = np.zeros((nch, N + 7))
    Yp[:, :N] = Y.T
    padded = np.zeros_like(full)
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_window_matrix_sums(ctx.h, Yp.ctypes.data_as(C.c_void_p), nch, N + 7,
                                                 t.ctypes.data_as(C.c_void_p), N, f.ctypes.data_as(C.c_void_p), len(f),
                                                 W.ctypes.data_as(C.c_void_p), n, nov, 1e-10, 0, K,
                                                 padded.ctypes.data_as(C.c_void_p), C.byref(info)))
    assert np.array_equal(padded, full)
    # window ranges add up (what sharded ranks all-reduce)
    a = lp.window_matrix_sums(Y, t, f, W, n, nov, 1e-10, 0, 11, ctx=ctx)
    b = lp.window_matrix_sums(Y, t, f, W, n, nov, 1e-10, 11, K, ctx=ctx)
    assert np.abs(a + b - full).max() <= 1e-14 * np.abs(full).max()
    # the coherence diagonal is exactly 1
    Co, _ = lp.ls_cohere_matrix(Y, t, f, nw=N // n, ctx=ctx)
    assert np.all(np.einsum("fii->fi", Co) == 1.0)


def test_singular_window_jitter_and_not_spd(ctx):
    """Window 2 sits at t = 0 throughout with f0 = 0: its -sin block is identically zero, so with lam = 0 its Cholesky
    breaks down.  Default options: the window is re-factorised alone with the jitter ridge (LPVS_INFO_JITTER), the others
    are untouched.  LPVS_OPT_JITTER = 0: LPVS_E_NOT_SPD naming window 2."""
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    N, nch, n = 3000, 3, 500
    t, Y = record(N, nch, seed=9)
    f = np.arange(64) * 2.0 / (t[n] - t[0])
    t[2 * n:3 * n] = 0.0
    W = o.hanning(n)
    sums = np.zeros((len(f), nch, nch), dtype=np.complex128)
    Yc = np.ascontiguousarray(Y.T)
    K = lp.window_count(N, n, 0)
    info = C.c_int(0)

    def call():
        return ctx.lib.lpvs_ls_window_matrix_sums(ctx.h, Yc.ctypes.data_as(C.c_void_p), nch, N, t.ctypes.data_as(C.c_void_p),
                                                  N, f.ctypes.data_as(C.c_void_p), len(f), W.ctypes.data_as(C.c_void_p), n,
                                                  0, 0.0, 0, K, sums.ctypes.data_as(C.c_void_p), C.byref(info))

    assert call() == L.OK and info.value == L.INFO_JITTER
    assert np.all(np.isfinite(sums))
    # the two-channel path takes the same retry on the same window.  The re-factorised window's answer is only defined to
    # cond(G + jitter ridge) eps, O(1) here (the ridge is Nreg eps max diag G on a rank-one block), hence the cond bar
    two = lp.window_sums(L.WIN_CSD, Y[:, 0], Y[:, 1], t, f, W, n, 0, 0.0, 0, K, ctx=ctx)
    assert rel(sums[:, 0, 1], two[:len(f)] + 1j * two[len(f):]) <= bar(_jitter_cond(t, f, n, W, lam=0.0))
    ctx.set_option(L.OPT_JITTER, 0)
    try:
        rc = call()
        msg = ctx.lib.lpvs_last_error(ctx.h).decode()
    finally:
        ctx.set_option(L.OPT_JITTER, 1)
    assert rc == L.E_NOT_SPD and info.value > 0 and "window 2 " in msg, (rc, info.value, msg)


def _jitter_cond(t, f, n, W, lam):
    """The largest cond of what the windows (noverlap = 0) are solved with: G + lam I, or G + max(lam, Nreg eps max diag G) I
    for a window whose factorisation breaks down."""
    worst = 1.0
    for k in range(len(t) // n):
        A, _ = o.get_fourier_regressor(t[k * n:(k + 1) * n], f)
        G = (A.T * W) @ A
        M = G + lam * np.eye(len(G))
        try:
            np.linalg.cholesky(M)
        except np.linalg.LinAlgError:
            M = G + max(lam, len(G) * EPS * np.diag(G).max()) * np.eye(len(G))
        worst = max(worst, np.linalg.cond(M))
    return worst


def test_jitter_retry_of_every_window(ctx):
    """A negative ridge makes the factorisation of EVERY window break down at its first pivot, so each window is re-done
    alone (re-factorised with max(lam, Nreg eps max diag G), its C right-hand sides solved against the new factor and
    written back to its own slot).  Here the re-factorised problems are well conditioned, so every entry must match the
    two-channel path, which takes the same retry, to the cond bar."""
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    N, nch, n = 3000, 3, 500
    t, Y = record(N, nch, seed=13)
    f = np.arange(64) * 2.0 / (t[n] - t[0])
    W = o.hanning(n)
    K = lp.window_count(N, n, 0)
    Yc = np.ascontiguousarray(Y.T)
    sums = np.zeros((len(f), nch, nch), dtype=np.complex128)
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_window_matrix_sums(ctx.h, Yc.ctypes.data_as(C.c_void_p), nch, N, t.ctypes.data_as(C.c_void_p), N,
                                                 f.ctypes.data_as(C.c_void_p), len(f), W.ctypes.data_as(C.c_void_p), n, 0,
                                                 -10.0, 0, K, sums.ctypes.data_as(C.c_void_p), C.byref(info)))
    assert info.value == L.INFO_JITTER
    tol = bar(_jitter_cond(t, f, n, W, lam=-10.0))
    assert tol < 1e-9
    for i in range(nch):
        psd = lp.window_sums(L.WIN_PSD, Y[:, i], None, t, f, W, n, 0, -10.0, 0, K, ctx=ctx)
        assert rel(sums[:, i, i].real, psd) <= tol
        for j in range(i + 1, nch):
            two = lp.window_sums(L.WIN_CSD, Y[:, i], Y[:, j], t, f, W, n, 0, -10.0, 0, K, ctx=ctx)
            assert rel(sums[:, i, j], two[:len(f)] + 1j * two[len(f):]) <= tol, (i, j)


def test_errors_and_edge_cases(ctx):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    N, nch, n = 2000, 3, 400
    t, Y = record(N, nch, seed=2)
    f = np.arange(20) * 2.0 / (t[n] - t[0])
    W = o.hanning(n)
    Yc = np.ascontiguousarray(Y.T)
    sums = np.zeros((len(f), nch, nch), dtype=np.complex128)
    info = C.c_int(0)

    def call(Ybuf, C_, ldY, nov=-1):
        return ctx.lib.lpvs_ls_window_matrix_sums(ctx.h, Ybuf.ctypes.data_as(C.c_void_p), C_, ldY, t.ctypes.data_as(C.c_void_p),
                                                  N, f.ctypes.data_as(C.c_void_p), len(f), W.ctypes.data_as(C.c_void_p), n,
                                                  nov, 1e-10, 0, 1, sums.ctypes.data_as(C.c_void_p), C.byref(info))

    assert call(Yc, 0, N) == L.E_BAD_ARG
    assert call(Yc, nch, N - 1) == L.E_BAD_ARG
    assert call(Yc, nch, N, nov=n) == L.E_BAD_ARG
    Yb = Yc.copy()
    Yb[1, 17] = np.nan
    assert call(Yb, nch, N) == L.E_NONFINITE
    assert call(Yc, nch, N) == L.OK  # the context stays usable
    with pytest.raises(ValueError):
        lp.window_matrix_sums(Y, t, f, W, n, -1, 1e-10, 0, 99, ctx=ctx)  # window range out of bounds
    with pytest.raises(TypeError):
        lp.ls_windowcsd_matrix(Y, t, f, estimator=lp.ls_sparse_spectral, ctx=ctx)
    with pytest.raises(TypeError):
        lp.ls_cohere_matrix(Y, t, f, window_func=lp.rect, ctx=ctx)
    # K = 0: empty sums finalise to NaN
    empty = lp.window_matrix_sums(Y, t, f, W, n, -1, 1e-10, 0, 0, ctx=ctx)
    assert not empty.any() and np.all(np.isnan(lp.window_matrix_finalize(L.WIN_CSD, empty, 0)))
    # Float32 in, Float32 / ComplexF32 out: the FP64 answer on the same inputs, rounded
    Y32, t32 = Y.astype(np.float32), t.astype(np.float32)
    S32, _ = lp.ls_windowcsd_matrix(Y32, t32, f, nw=5, ctx=ctx)
    S64, _ = lp.ls_windowcsd_matrix(Y32.astype(np.float64), t32.astype(np.float64), f, nw=5, ctx=ctx)
    assert S32.dtype == np.complex64 and np.array_equal(S32, S64.astype(np.complex64))
    P32, _ = lp.ls_windowpsd_multi(Y32, t32, f, nw=5, ctx=ctx)
    C32, _ = lp.ls_cohere_matrix(Y32, t32, f, nw=5, ctx=ctx)
    assert P32.dtype == np.float32 and C32.dtype == np.float32
