"""GPU: ls_spectral of C channels at shared sample times (lpvs_ls_spectral_multi[_dev]) against the oracle, the single-channel
call, and its exact properties.

Every channel is scaled by 10^((c mod 7) - 3) and judged against its own norm, so a quiet channel cannot hide behind a loud
one.  Bars as tests/test_gpu_rankdef.py: max(1e-9, 50 cond([A; lam I]) eps) unweighted (against the SVD and the QR solve of
the same matrix), max(1e-9, 40 cond(A'WA + lam I) eps) weighted."""
import ctypes as C

import numpy as np
import pytest
import scipy.linalg as sla

from oracle import lpvs_oracle as o

pytestmark = pytest.mark.gpu

EPS = np.finfo(float).eps


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(b)


def scale(c):
    return 10.0 ** ((c % 7) - 3)


def signal(N, seed, T=10.0):
    rng = np.random.default_rng(seed)
    t = np.sort(T * rng.random(N))
    y = np.sin(2 * np.pi * 20 * t) + 0.5 * np.cos(2 * np.pi * 55 * t + 1) + 0.1 * rng.standard_normal(N)
    return t, y


def channels(t, nch, seed):
    """Resolved sinusoids, white noise and mixtures, each scaled by 10^((c mod 7) - 3)."""
    rng = np.random.default_rng(seed)
    Y = np.empty((len(t), nch))
    for c in range(nch):
        k = c % 3
        if k == 0:
            y = np.sin(2 * np.pi * (5 + 3 * c) * t + c) + 0.05 * rng.standard_normal(len(t))
        elif k == 1:
            y = rng.standard_normal(len(t))
        else:
            y = np.cos(2 * np.pi * 17 * t) + 0.5 * rng.standard_normal(len(t))
        Y[:, c] = scale(c) * y
    return Y


def svd_qr_solutions(A, Y, lam, zf, literal=True):
    """svd([A; lam I]) \\ [Y; 0] (Julia's rule, as oracle.svd_solve) and the QR solve, every column at once."""
    n = A.shape[1]
    M = np.vstack([A, lam * np.eye(n)])
    R = np.vstack([Y, np.zeros((n, Y.shape[1]))])
    Q, Rq = np.linalg.qr(M)
    xq = sla.solve_triangular(Rq, Q.T @ R, check_finite=False)
    xs = None
    if literal:
        U, s, Vt = sla.svd(M, full_matrices=False, lapack_driver="gesdd")
        k = int(np.sum(s > EPS * s[0]))
        xs = Vt[:k].T @ ((U[:, :k].T @ R) / s[:k, None])
        xs = np.stack([o.fourier2complex(xs[:, c], zf) for c in range(Y.shape[1])], axis=1)
    xq = np.stack([o.fourier2complex(xq[:, c], zf) for c in range(Y.shape[1])], axis=1)
    return xs, xq


def cond_aug(A, lam):
    s = np.linalg.svd(A, compute_uv=False)
    smin = s[-1] if A.shape[0] >= A.shape[1] else 0.0
    return np.hypot(s[0], lam) / np.hypot(smin, lam)


def check_unweighted(X, t, f, Y, lam=1e-10, literal=True, cm=None):
    A, zf = o.get_fourier_regressor(t, f)
    cm = cond_aug(A, lam) if cm is None else cm
    tol = max(1e-9, 50.0 * cm * EPS)
    xs, xq = svd_qr_solutions(A, Y, lam, zf, literal)
    worst = 0.0
    for c in range(Y.shape[1]):
        e = rel(X[:, c], xq[:, c])
        if literal:
            e = max(e, rel(X[:, c], xs[:, c]))
        worst = max(worst, e / tol)
    print(f"unweighted N={len(t)} Nf={len(f)} C={Y.shape[1]}: cond {cm:.2e} worst/bar {worst:.3f}")
    assert worst <= 1.0
    return xq


def multi(ctx, Y, t, f, W=None, lam=1e-10):
    import lpvspectral_jl_b200 as lp

    X, _, info = lp.ls_spectral_multi(Y, t, f, W, lam=lam, ctx=ctx, return_info=True)
    return X, info


def single_infos(ctx, Y, t, f, W=None, lam=1e-10):
    import lpvspectral_jl_b200 as lp

    xs, infos = [], []
    for c in range(Y.shape[1]):
        x, _, i = lp.ls_spectral(Y[:, c], t, f, W, lam=lam, ctx=ctx, return_info=True)
        xs.append(x)
        infos.append(i)
    return np.stack(xs, axis=1), np.array(infos)


def dev_call(ctx, Y, t, f, W=None, lam=1e-10, ldY=None):
    """lpvs_ls_spectral_multi_dev on device copies of Y (channel c at c ldY), t and W."""
    import torch

    dev = torch.device("cuda", ctx.device)
    N, nch = Y.shape
    ldY = N if ldY is None else ldY
    Yp = np.zeros((nch, ldY))
    Yp[:, :N] = Y.T
    Yd = torch.from_numpy(Yp).to(dev)
    td = torch.from_numpy(np.ascontiguousarray(t, dtype=np.float64)).to(dev)
    Wd = None if W is None else torch.from_numpy(np.ascontiguousarray(W, dtype=np.float64)).to(dev)
    torch.cuda.synchronize(dev)
    f = np.ascontiguousarray(f, dtype=np.float64)
    X = np.empty((nch, len(f)), dtype=np.complex128)
    info = np.zeros(nch, dtype=np.int32)
    ctx.check(ctx.lib.lpvs_ls_spectral_multi_dev(ctx.h, C.c_void_p(Yd.data_ptr()), nch, ldY, C.c_void_p(td.data_ptr()), N,
                                                 f.ctypes.data_as(C.c_void_p), len(f),
                                                 None if Wd is None else C.c_void_p(Wd.data_ptr()), lam,
                                                 X.ctypes.data_as(C.c_void_p), info.ctypes.data_as(C.POINTER(C.c_int))))
    return X.T, info


# ---- parity ------------------------------------------------------------------------------------------------------------


def test_reference_kat_in_every_column(ctx):
    """test/runtests.jl:186-188 (t = 0:0.1:99.9, default freqs, 1000 x 1001) in every column, scaled per channel."""
    import lpvspectral_jl_b200 as lp

    t = np.arange(1000) * 0.1
    y = np.sin(2 * np.pi * t)
    nch = 4
    Y = np.stack([scale(c) * y for c in range(nch)], axis=1)
    X, f, info = lp.ls_spectral_multi(Y, t, ctx=ctx, return_info=True)
    _, i1, = single_infos(ctx, Y[:, :1], t, f)
    assert list(info) == [i1[0]] * nch
    A, zf = o.get_fourier_regressor(t, f)
    xs, xq = svd_qr_solutions(A, Y, 1e-10, zf)
    for c in range(nch):
        a = np.abs(X[:, c] / scale(c)) ** 2
        assert a.argmax() + 1 == 101 and abs(a.max() - 2.0 * len(f)) < 1e-4
        assert rel(X[:, c], xq[:, c]) <= 1e-9
        assert rel(X[:, c], xs[:, c]) <= 1e-6


@pytest.mark.parametrize("N,frac,nch", [(1000, None, 5), (4096, 0.25, 6), (1024, 0.5, 5), (1024, 0.36, 6), (1024, 0.40, 6)])
def test_parity_unweighted(ctx, N, frac, nch):
    """The default call (Nreg = N+1), PARITY-1 (4096 x 1024: info 0), cfg1's shape at N = 1024 (info QR) and the
    cond(A) ~ 1e5..1e7 band; every channel against the SVD and QR solves, and its info against the single call's."""
    t, _ = signal(N, 1)
    f = o.default_freqs(t)
    if frac is not None:
        f = f[: int(N * frac)]
    Y = channels(t, nch, N)
    X, info = multi(ctx, Y, t, f)
    _, info1 = single_infos(ctx, Y, t, f)
    print(f"N={N} frac={frac}: info {list(info)} single {list(info1)}")
    assert list(info) == list(info1)
    if frac == 0.25:
        assert list(info) == [0] * nch
    if frac == 0.5:
        assert all(i == 2 for i in info)
    check_unweighted(X, t, f, Y)


def test_cfg1_full_size(ctx):
    """BASELINE configs[0]: N = 4096 irregular samples, 2048 freqs, lam = 1e-10: every channel on the QR route."""
    from lpvspectral_jl_b200 import _lib as L

    t, _ = signal(4096, 1)
    f = o.default_freqs(t)[:2048]
    Y = channels(t, 3, 11)
    X, info = multi(ctx, Y, t, f)
    assert list(info) == [L.INFO_QR] * 3
    A, _ = o.get_fourier_regressor(t, f)
    check_unweighted(X, t, f, Y, literal=False, cm=np.linalg.norm(A, 2) / 1e-10)  # the literal SVD takes minutes here


@pytest.mark.parametrize("uniform", [True, False])
def test_parity_weighted_hann(ctx, uniform):
    import lpvspectral_jl_b200 as lp

    N = 1500
    t = np.arange(N) * 0.01 if uniform else signal(N, 5)[0]
    f = o.default_freqs(t)[:300]
    W = lp.hanning(N)
    Y = channels(t, 7, 21)
    X, info = multi(ctx, Y, t, f, W)
    X1, info1 = single_infos(ctx, Y, t, f, W)
    assert list(info) == list(info1)
    A, _ = o.get_fourier_regressor(t, f)
    G = (A.T * W) @ A + 1e-10 * np.eye(A.shape[1])
    tol = max(1e-9, 40.0 * np.linalg.cond(G) * EPS)
    for c in range(Y.shape[1]):
        xr, _ = o.ls_spectral(Y[:, c], t, f, W, mode="literal")
        assert rel(X[:, c], xr) <= tol, (c, rel(X[:, c], xr), tol)
        assert rel(X[:, c], X1[:, c]) <= tol


# ---- routes --------------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("N,frac", [(1024, 0.36), (1024, 0.40), (1024, 0.45)])
def test_route_flags_match_the_single_call(ctx, N, frac):
    """Sinusoids, white noise and a zero channel side by side: each channel takes the route its single call takes."""
    t, _ = signal(N, 1)
    f = o.default_freqs(t)[: int(N * frac)]
    rng = np.random.default_rng(3)
    Y = np.stack([np.sin(2 * np.pi * 7 * t) + np.cos(2 * np.pi * 31 * t), rng.standard_normal(N), np.zeros(N),
                  1e3 * np.sin(2 * np.pi * 12 * t)], axis=1)
    X, info = multi(ctx, Y, t, f)
    X1, info1 = single_infos(ctx, Y, t, f)
    print(f"routes frac={frac}: {list(info)}")
    assert list(info) == list(info1)
    assert np.all(X[:, 2] == 0)
    A, zf = o.get_fourier_regressor(t, f)
    tol = max(1e-9, 50.0 * cond_aug(A, 1e-10) * EPS)
    _, xq = svd_qr_solutions(A, Y, 1e-10, zf, literal=False)
    for c in (0, 1, 3):
        assert rel(X[:, c], xq[:, c]) <= tol and rel(X[:, c], X1[:, c]) <= 2 * tol


# ---- edges ---------------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("nch", [1, 2, 8, 9, 16, 17, 32, 33])
def test_channel_counts(ctx, nch):
    t, _ = signal(300, 2)
    f = o.default_freqs(t)[:100]
    Y = channels(t, nch, nch)
    X, info = multi(ctx, Y, t, f)
    check_unweighted(X, t, f, Y)
    # a channel alone gives the bits it has inside the call
    for c in sorted({0, nch // 2, nch - 1}):
        Xc, ic = multi(ctx, Y[:, c:c + 1], t, f)
        assert np.array_equal(Xc[:, 0], X[:, c]) and ic[0] == info[c]


@pytest.mark.parametrize("Nf,zero", [(40, True), (40, False), (100, True), (100, False), (700, True)])
def test_block_counts_and_zero_frequency(ctx, Nf, zero):
    """nb = 1, 2 and many, with and without a zero first frequency (Nf = 700 > N / 2: the dual route)."""
    t, _ = signal(1200, 3)
    df = 0.5 / (t[-1] - t[0]) * len(t) / 700
    f = (np.arange(Nf) + (0 if zero else 1)) * df
    Y = channels(t, 5, Nf)
    X, info = multi(ctx, Y, t, f)
    _, info1 = single_infos(ctx, Y, t, f)
    # cond(A) ~ 1e7 puts the first refinement step at the 0.05 contraction test: a channel's first iterate (explicit L^-1
    # here, substitution in the single call) can tip it to the other route.  Both routes meet the bar.
    print(f"Nf={Nf} zero={zero}: info {list(info)} single {list(info1)}")
    check_unweighted(X, t, f, Y)


def test_tiny_N_and_padded_ldY(ctx):
    t = np.array([0.0, 0.13, 0.31, 0.47, 0.52])
    f = np.array([0.0, 0.5, 1.1])
    Y = channels(t, 3, 0)
    X, info = multi(ctx, Y, t, f)
    check_unweighted(X, t, f, Y)
    Xd, infod = dev_call(ctx, Y, t, f, ldY=len(t) + 7)
    assert np.array_equal(Xd, X) and list(infod) == list(info)


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4, 5])
def test_weighted_phase_modes(ctx, mode):
    """Every phase mode on the weighted path agrees with the single-channel call in that mode (uniform grid)."""
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    N = 2048
    t = np.arange(N) * 0.01
    f = np.arange(150) * (1.0 / (N * 0.01))
    W = lp.hanning(N)
    Y = channels(t, 9, 5)
    ctx.set_option(L.OPT_PHASE_MODE, mode)
    try:
        X, info = multi(ctx, Y, t, f, W)
        X1, info1 = single_infos(ctx, Y, t, f, W)
    finally:
        ctx.set_option(L.OPT_PHASE_MODE, 0)
    assert list(info) == list(info1)
    # the structured modes form G from trigonometric sums, the right-hand sides from the chains (as the matrix path does)
    tol = 1e-9 if mode < L.PHASE_STRUCTURED else 1e-6
    for c in range(Y.shape[1]):
        e = rel(X[:, c], X1[:, c])
        print(f"mode {mode} channel {c}: {e:.2e}")
        assert e <= tol, (mode, c, e)


# ---- exact properties ----------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("weighted,N,frac", [(False, 1000, None), (False, 1024, 0.25), (False, 1024, 0.4),
                                             (False, 1024, 0.5), (True, 1024, 0.3)])
def test_exact_properties(ctx, weighted, N, frac):
    import lpvspectral_jl_b200 as lp

    t, _ = signal(N, 9)
    f = o.default_freqs(t)
    if frac is not None:
        f = f[: int(N * frac)]
    W = lp.hanning(N) if weighted else None
    Y = channels(t, 33, 4)
    Y[:, 5] = Y[:, 2]  # identical channels
    Y[:, 7] = 0.0      # a zero channel
    X, info = multi(ctx, Y, t, f, W)
    assert np.array_equal(X[:, 5], X[:, 2]) and info[5] == info[2]
    assert np.all(X[:, 7] == 0)
    perm = np.random.default_rng(0).permutation(33)
    Xp, infop = multi(ctx, Y[:, perm], t, f, W)
    assert np.array_equal(Xp, X[:, perm]) and np.array_equal(infop, info[perm])
    for c in (0, 13, 32):
        Xc, ic = multi(ctx, Y[:, c:c + 1], t, f, W)
        assert np.array_equal(Xc[:, 0], X[:, c]) and ic[0] == info[c]
    # the zero channel changes no other column's bits
    keep = [c for c in range(33) if c != 7]
    Xz, infoz = multi(ctx, Y[:, keep], t, f, W)
    assert np.array_equal(Xz, X[:, keep]) and np.array_equal(infoz, info[keep])
    Xd, infod = dev_call(ctx, Y, t, f, W, ldY=N + 3)
    assert np.array_equal(Xd, X) and np.array_equal(infod, info)


# ---- errors and jitter ---------------------------------------------------------------------------------------------------


def test_errors(ctx):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    t, _ = signal(200, 1)
    f = o.default_freqs(t)[:40]
    Y = channels(t, 6, 1)
    Yc = np.ascontiguousarray(Y.T)
    X = np.empty((6, 40), dtype=np.complex128)
    info = np.zeros(6, dtype=np.int32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    ip = info.ctypes.data_as(C.POINTER(C.c_int))
    assert ctx.lib.lpvs_ls_spectral_multi(ctx.h, vp(Yc), 0, 200, vp(t), 200, vp(f), 40, None, 1e-10, vp(X), ip) == L.E_BAD_ARG
    assert ctx.lib.lpvs_ls_spectral_multi(ctx.h, vp(Yc), 6, 199, vp(t), 200, vp(f), 40, None, 1e-10, vp(X), ip) == L.E_BAD_ARG
    assert ctx.lib.lpvs_ls_spectral_multi(ctx.h, None, 6, 200, vp(t), 200, vp(f), 40, None, 1e-10, vp(X), ip) == L.E_BAD_ARG
    Yn = Y.copy()
    Yn[17, 4] = np.nan
    Yn[3, 5] = np.inf
    with pytest.raises(lp.LpvsError, match="channel 4"):
        lp.ls_spectral_multi(Yn, t, f, ctx=ctx)
    with pytest.raises(ValueError):
        lp.ls_spectral_multi(Y, t[:-1], f, ctx=ctx)
    with pytest.raises(ValueError):
        lp.ls_spectral_multi(Y, t, f, np.ones(199), ctx=ctx)
    # the context is still usable
    X2, _ = multi(ctx, Y, t, f)
    check_unweighted(X2, t, f, Y)


def test_weighted_singular_gram_jitters_every_channel(ctx):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    N = 600
    t, _ = signal(N, 6)
    f = np.repeat(np.arange(1, 41) * 0.5, 2)  # every column twice: A'WA exactly singular
    W = lp.hanning(N)
    Y = channels(t, 5, 6)
    X, info = multi(ctx, Y, t, f, W, lam=0.0)  # a ridge lam >> Nreg eps max diag would keep the factor positive
    X1, info1 = single_infos(ctx, Y, t, f, W, lam=0.0)
    assert list(info) == [L.INFO_JITTER] * 5 and list(info1) == [L.INFO_JITTER] * 5
    assert np.all(np.isfinite(X))
    # both are (A'WA + jitter I)^-1 A'Wy with cond ~ 1 / (Nreg eps): they agree only to that condition number
    print("jitter: multi vs single", [f"{rel(X[:, c], X1[:, c]):.1e}" for c in range(5)])
