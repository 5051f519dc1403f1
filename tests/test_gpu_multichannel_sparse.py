"""GPU: sparse cross-spectral matrices (lpvs_ls_window_matrix_sparse_sums[_dev], k_admm_multi) against the sparse matrix
oracle of tests/oracle_matrix_sparse.py, against the two-channel sparse path, and their exact properties.

Chunk classes of k_admm_multi (csrc/admm.cu admm_multi_plan): CC = 8 for C <= 8, 16 for C <= 16, 32 above, narrowed while
CC (Np + 4) doubles of right-hand sides do not fit next to the ring: CC = 32 up to Np = 512, 16 up to 1024, 8 up to 2176,
and above that CC = 8 with the right-hand sides in global memory.  C in {1, 2, 3, 8, 9, 17, 33} runs every class with full
and partial last chunks; Nf = 256 / 300 / 512 / 576 / 1088 / 1100 puts Np on both sides of every switch.  -m gpu."""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle import lpvs_oracle as o

import oracle_matrix_sparse as oms

pytestmark = pytest.mark.gpu

MODES = {"auto": 0, "chain": 1, "direct": 2, "chain_ref": 3, "structured": 4, "structured_ref": 5}
PROX = {"l1": (o.NormL1(0.4), 0.4), "l0": (o.NormL0(0.01), 0.01), "ball": (o.IndBallL0(6), 6)}
KW = dict(mu=0.05, iters=4000, tol=1e-10)


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def record(N, nch, seed, T=10.0):
    """Every channel its own tone plus a shared one and white noise; channel c scaled by 10^((c mod 5) - 2)."""
    rng = np.random.default_rng(seed)
    t = np.sort(T * rng.random(N))
    common = np.sin(2 * np.pi * 1.3 * t)
    Y = np.stack([(0.3 + 0.1 * c) * common + np.cos(2 * np.pi * (0.7 + 0.23 * c) * t + c)
                  + 0.3 * rng.standard_normal(N) for c in range(nch)], axis=1)
    return t, Y * 10.0 ** ((np.arange(nch) % 5) - 2.0)


def lib_prox(name, scale=1.0):
    import lpvspectral_jl_b200 as lp

    pg = PROX[name][0]
    if name == "l1":
        return lp.NormL1(pg.lam * scale), o.NormL1(pg.lam * scale)
    if name == "l0":
        return lp.NormL0(pg.lam * scale), o.NormL0(pg.lam * scale)
    return lp.IndBallL0(pg.r), pg


def set_mode(ctx, mode):
    from lpvspectral_jl_b200 import _lib as L

    ctx.check(ctx.lib.lpvs_set_option(ctx.h, L.OPT_PHASE_MODE, float(MODES[mode])))


def set_batch(ctx, b):
    from lpvspectral_jl_b200 import _lib as L

    ctx.check(ctx.lib.lpvs_set_option(ctx.h, L.OPT_WINDOW_BATCH, float(b)))


@pytest.fixture
def mctx(ctx):
    yield ctx
    set_mode(ctx, "auto")
    set_batch(ctx, 0)


def check_entries(S, R, bar=1e-8):
    fin = np.isfinite(R)
    assert np.array_equal(np.isfinite(S), fin)
    assert np.linalg.norm((S - R)[fin]) <= bar * np.linalg.norm(R[fin])
    d = np.abs(np.einsum("fii->fi", R))
    scale = np.sqrt(d[:, :, None] * d[:, None, :])
    assert np.all(np.abs(S - R) <= bar * scale + 1e-300)


def sums(ctx, Y, t, f, W, n, nov, pk, pp, k0, k1, mu=0.05, iters=4000, tol=1e-10):
    from lpvspectral_jl_b200 import _lib as L

    pk = {"l1": L.PROX_L1, "l0": L.PROX_L0, "ball": L.PROX_BALL_L0}.get(pk, pk)
    nch = Y.shape[1]
    S = np.zeros((len(f), nch, nch), dtype=np.complex128)
    its = np.zeros((max(k1 - k0, 1), nch), dtype=np.int64)
    res = np.zeros((max(k1 - k0, 1), nch))
    Yc = np.ascontiguousarray(Y.T)
    info = C.c_int(0)
    rc = ctx.lib.lpvs_ls_window_matrix_sparse_sums(ctx.h, vp(Yc), nch, Y.shape[0], vp(t), len(t), vp(f), len(f), vp(W), n,
                                                   nov, pk, float(pp), mu, iters, tol, k0, k1, vp(S), vp(its), vp(res),
                                                   C.byref(info))
    return rc, S, its, res


def dev_sums(ctx, Y, t, f, W, n, nov, pk, pp, k0, k1, ldY, mu=0.05, iters=4000, tol=1e-10):
    import torch
    from lpvspectral_jl_b200 import _lib as L

    pk = {"l1": L.PROX_L1, "l0": L.PROX_L0, "ball": L.PROX_BALL_L0}[pk]
    dev = torch.device("cuda", ctx.device)
    N, nch = Y.shape
    Yp = np.zeros((nch, ldY))
    Yp[:, :N] = Y.T
    Yd = torch.from_numpy(Yp).to(dev)
    td = torch.from_numpy(t).to(dev)
    torch.cuda.synchronize(dev)
    S = np.zeros((len(f), nch, nch), dtype=np.complex128)
    its = np.zeros((k1 - k0, nch), dtype=np.int64)
    res = np.zeros((k1 - k0, nch))
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_window_matrix_sparse_sums_dev(ctx.h, C.c_void_p(Yd.data_ptr()), nch, ldY,
                                                            C.c_void_p(td.data_ptr()), N, vp(f), len(f), vp(W), n, nov, pk,
                                                            float(pp), mu, iters, tol, k0, k1, vp(S), vp(its), vp(res),
                                                            C.byref(info)))
    return S, its, res


# name: (C, Nf, zero first frequency, n, nw, noverlap, non-uniform)
SHAPES = {
    "c1_nf20_f0zero": (1, 20, True, 211, 3, "half", False),
    "c2_nf17": (2, 17, False, 187, 3, "zero", False),
    "c3_nf24_hop1": (3, 24, False, 97, 2, "n-1", False),
    "c8_nf20_f0zero": (8, 20, True, 203, 3, "half", False),
    "c9_nf33": (9, 33, False, 229, 2, "zero", False),
    "c17_nf20": (17, 20, False, 173, 2, "half", False),
    "c33_nf12_f0zero": (33, 12, True, 131, 2, "half", False),
    "c9_nf20_nonuniform": (9, 20, False, 203, 2, "half", True),
}
CASES = [(s, m, p) for s in SHAPES for m in (("auto", "direct") if SHAPES[s][6] else ("auto", "direct", "chain_ref"))
         for p in PROX]


def grid(Nf, f0zero, Tw, nonuniform):
    if nonuniform:
        f = np.cumsum(1.0 + 0.5 * np.random.default_rng(Nf).random(Nf)) * 0.5 / Tw
        return np.concatenate([[0.0], f[:-1]]) if f0zero else f
    return (np.arange(Nf) + (0 if f0zero else 1)) * 0.5 / Tw


@functools.lru_cache(maxsize=None)
def shape_case(name, prox):
    nch, Nf, f0zero, n, nw, nov, nonuni = SHAPES[name]
    N = nw * n + nw - 1
    t, Y = record(N, nch, seed=N + nch)
    noverlap = {"half": n >> 1, "zero": 0, "n-1": n - 1}[nov]
    f = grid(Nf, f0zero, t[n] - t[0], nonuni)
    pg = PROX[prox][0]
    S, K, _, its, res = oms.sparse_matrix_sums(Y, t, f, nw=nw, noverlap=noverlap, window_func=o.hanning, proxg=pg, **KW)
    return t, Y, f, n, nw, noverlap, S, K, its


@pytest.mark.parametrize("shape,mode,prox", CASES)
def test_against_sparse_oracle(mctx, shape, mode, prox):
    import lpvspectral_jl_b200 as lp

    t, Y, f, n, nw, noverlap, R, K, _ = shape_case(shape, prox)
    set_mode(mctx, mode)
    pg = lib_prox(prox)[0]
    S, _ = lp.ls_sparse_windowcsd_matrix(Y, t, f, nw=nw, noverlap=noverlap, window_func=lp.hanning, proxg=pg, ctx=mctx,
                                         **KW)
    Rn = (R.real / K) + 1j * (R.imag / K)
    check_entries(S, Rn)
    P, _ = lp.ls_sparse_windowpsd_multi(Y, t, f, nw=nw, noverlap=noverlap, window_func=lp.hanning, proxg=pg, ctx=mctx,
                                        **KW)
    Pr = np.einsum("fii->fi", R).real / float(K) ** 2
    assert np.linalg.norm(P - Pr) <= 1e-8 * np.linalg.norm(Pr)
    assert np.all(np.abs(P - Pr) <= 1e-8 * Pr + 1e-300)
    assert mctx.last_window_iters.shape == (K, Y.shape[1])
    Co, _ = lp.ls_sparse_cohere_matrix(Y, t, f, nw=nw, noverlap=noverlap, proxg=pg, ctx=mctx, **KW)
    Cr, _ = oms.ls_sparse_cohere_matrix(Y, t, f, nw=nw, noverlap=noverlap, proxg=PROX[prox][0], **KW)
    assert np.array_equal(np.isnan(Co), np.isnan(Cr))
    fin = np.isfinite(Cr)
    assert np.all(np.abs(Co[fin] - Cr[fin]) <= 1e-7 * np.maximum(np.abs(Cr[fin]), 1e-3))


@pytest.mark.parametrize("mode", list(MODES))
def test_against_two_channel_path(mctx, mode):
    import lpvspectral_jl_b200 as lp

    t, Y = record(3 * 301 + 2, 3, 5)
    n, nov = 301, 150
    f = np.arange(1, 30) * 0.5 / (t[n] - t[0])
    set_mode(mctx, mode)
    kw = dict(proxg=lp.NormL1(0.05), **KW)
    S, _ = lp.ls_sparse_windowcsd_matrix(Y, t, f, nw=3, noverlap=nov, window_func=lp.hanning, ctx=mctx, **kw)
    its = mctx.last_window_iters.copy()
    P, _ = lp.ls_sparse_windowpsd_multi(Y, t, f, nw=3, noverlap=nov, window_func=lp.hanning, ctx=mctx, **kw)
    K = lp.window_count(len(t), n, nov)
    W = lp.hanning(n)
    for i in range(3):
        Pi, _ = lp.ls_windowpsd(Y[:, i], t, f, nw=3, noverlap=nov, window_func=lp.hanning,
                                estimator=lp.ls_sparse_spectral, ctx=mctx, **kw)
        assert np.linalg.norm(P[:, i] - Pi) <= 1e-8 * np.linalg.norm(Pi)
        _, it1, res1 = lp.window_sparse_sums(0, Y[:, i], None, t, f, W, n, nov, kw["proxg"], KW["mu"], KW["iters"],
                                             KW["tol"], 0, K, ctx=mctx, return_info=True)
        _, _, res_m = lp.window_matrix_sparse_sums(Y[:, i:i + 1], t, f, W, n, nov, kw["proxg"], KW["mu"], KW["iters"],
                                                   KW["tol"], 0, K, ctx=mctx, return_info=True)
        diff = np.abs(its[:, i] - it1[:, 0])
        assert diff.max() <= 1
        near = (np.abs(res1[:, 0] - KW["tol"]) <= 1e-3 * KW["tol"]) | (np.abs(res_m[:, 0] - KW["tol"]) <= 1e-3 * KW["tol"])
        assert np.all((diff == 0) | near)
        for j in range(3):
            Sij, _ = lp.ls_windowcsd(Y[:, i], Y[:, j], t, f, nw=3, noverlap=nov, window_func=lp.hanning,
                                     estimator=lp.ls_sparse_spectral, ctx=mctx, **kw)
            assert np.linalg.norm(S[:, i, j] - Sij) <= 1e-8 * np.sqrt(np.linalg.norm(S[:, i, i]) * np.linalg.norm(S[:, j, j]))


def _bits(a, b):
    """Bit for bit, except the sign of an exact zero: k_window_matrix_accum computes S_ij for i <= j and writes S_ji as its
    conjugate, so reordering the channels turns an imaginary +0 into -0 (sparse solutions have many exact zeros)."""
    a, b = np.ascontiguousarray(np.asarray(a) + 0), np.ascontiguousarray(np.asarray(b) + 0)
    return np.array_equal(a.view(np.uint8), b.view(np.uint8))


@pytest.mark.parametrize("mode", ["auto", "structured_ref"])
@pytest.mark.parametrize("prox", list(PROX))
def test_exact_properties(mctx, mode, prox):
    set_mode(mctx, mode)
    t, Y = record(2 * 211 + 5, 33, 11, T=20.0)
    n, nov = 211, 105
    f = np.arange(1, 21) * 0.5 / (t[n] - t[0])
    W = np.hanning(n)
    K = int(mctx.lib.lpvs_window_count(len(t), n, nov))
    pp = PROX[prox][1]
    rc, S, its, res = sums(mctx, Y, t, f, W, n, nov, prox, pp, 0, K)
    assert rc == 0
    # permuting the channels permutes S, the counts and the residuals bit for bit
    perm = np.random.default_rng(1).permutation(33)
    _, Sp, itp, rsp = sums(mctx, Y[:, perm], t, f, W, n, nov, prox, pp, 0, K)
    assert _bits(Sp, S[:, perm][:, :, perm]) and _bits(itp, its[:, perm]) and _bits(rsp, res[:, perm])
    # a pair alone gives the bits of that pair inside the C = 33 call
    for a, b in ((0, 32), (17, 5)):
        _, S2, it2, rs2 = sums(mctx, Y[:, [a, b]], t, f, W, n, nov, prox, pp, 0, K)
        assert _bits(S2, S[:, [a, b]][:, :, [a, b]]) and _bits(it2, its[:, [a, b]]) and _bits(rs2, res[:, [a, b]])
    # two identical channels: identical counts, coherence exactly 1 where S_ii != 0
    Yd = np.concatenate([Y[:, :3], Y[:, 2:3]], axis=1)
    _, Sd, itd, _ = sums(mctx, Yd, t, f, W, n, nov, prox, pp, 0, K)
    assert _bits(itd[:, 2], itd[:, 3])
    out = np.empty((len(f), 4, 4))
    mctx.lib.lpvs_ls_window_matrix_finalize(2, vp(Sd), len(f), 4, K, vp(out))
    nz = Sd[:, 2, 2].real != 0
    assert np.all(out[nz, 2, 3] == 1.0) and np.all(out[nz, 3, 2] == 1.0)
    # a zero channel: zero row and column, count 1, every other entry unchanged
    Yz = Y[:, :9].copy()
    Yz[:, 4] = 0.0
    _, S9, it9, _ = sums(mctx, Y[:, :9], t, f, W, n, nov, prox, pp, 0, K)
    _, Sz, itz, _ = sums(mctx, Yz, t, f, W, n, nov, prox, pp, 0, K)
    keep = [c for c in range(9) if c != 4]
    assert np.all(Sz[:, 4, :] == 0) and np.all(Sz[:, :, 4] == 0) and np.all(itz[:, 4] == 1)
    assert _bits(Sz[:, keep][:, :, keep], S9[:, keep][:, :, keep]) and _bits(itz[:, keep], it9[:, keep])
    # LPVS_OPT_WINDOW_BATCH in {1, 3, auto}: the same bits
    for b in (1, 3):
        set_batch(mctx, b)
        _, Sb, itb, rsb = sums(mctx, Y[:, :9], t, f, W, n, nov, prox, pp, 0, K)
        assert _bits(Sb, S9) and _bits(itb, it9)
    set_batch(mctx, 0)


def test_host_and_dev_forms_agree(mctx):
    t, Y = record(5 * 151, 10, 3)
    n, nov = 151, 75
    f = np.arange(0, 17) * 0.5 / (t[n] - t[0])
    W = np.hanning(n)
    K = int(mctx.lib.lpvs_window_count(len(t), n, nov))
    rc, S, its, res = sums(mctx, Y, t, f, W, n, nov, "l1", 0.3, 2, K)
    assert rc == 0
    Sd, itd, rsd = dev_sums(mctx, Y, t, f, W, n, nov, "l1", 0.3, 2, K, ldY=len(t) + 37)
    assert _bits(S, Sd) and _bits(its, itd) and _bits(res, rsd)


def test_budget_edges(mctx):
    t, Y = record(4 * 131, 5, 9)
    n, nov = 131, 65
    f = np.arange(1, 15) * 0.5 / (t[n] - t[0])
    W = np.hanning(n)
    K = int(mctx.lib.lpvs_window_count(len(t), n, nov))
    rc, S, its, _ = sums(mctx, Y, t, f, W, n, nov, "l1", 0.05, 0, K, iters=0)
    assert rc == 0 and np.all(S == 0) and np.all(its == 0)
    rc, S, its, res = sums(mctx, Y, t, f, W, n, nov, "l1", 0.05, 0, K, tol=np.inf)
    assert rc == 0 and np.all(its == 1) and np.any(S != 0)
    rc, S, its, res = sums(mctx, Y, t, f, W, n, nov, "l1", 0.05, 0, K, iters=300, tol=1e-7)
    assert rc == 0 and its.max() <= 300 and np.all(res[its < 300] < 1e-7)


# Nf -> Np: 256 -> 512, 300 -> 640, 512 -> 1024, 576 -> 1152, 1088 -> 2176, 1100 -> 2304
@pytest.mark.parametrize("Nf,nch", [(256, 33), (300, 33), (512, 17), (576, 17), (1088, 9), (1100, 9)])
def test_large_np_against_two_channel_path(mctx, Nf, nch):
    import lpvspectral_jl_b200 as lp

    n = 2 * Nf + 301
    t, Y = record(2 * n, nch, Nf, T=40.0)
    f = np.arange(1, Nf + 1) * 0.5 / (t[n] - t[0])
    kw = dict(proxg=lp.NormL1(0.05), mu=0.05, iters=300, tol=1e-10)
    S, _ = lp.ls_sparse_windowcsd_matrix(Y, t, f, nw=2, noverlap=0, window_func=lp.hanning, ctx=mctx, **kw)
    for i, j in ((0, nch - 1), (nch // 2, 1)):
        Sij, _ = lp.ls_windowcsd(Y[:, i], Y[:, j], t, f, nw=2, noverlap=0, window_func=lp.hanning,
                                 estimator=lp.ls_sparse_spectral, ctx=mctx, **kw)
        assert np.linalg.norm(S[:, i, j] - Sij) <= 1e-8 * np.sqrt(np.linalg.norm(S[:, i, i]) * np.linalg.norm(S[:, j, j]))


def test_errors(mctx):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    t, Y = record(3 * 101, 3, 4)
    n, nov = 101, 50
    f = np.arange(1, 9) * 0.5 / (t[n] - t[0])
    W = np.hanning(n)
    K = int(mctx.lib.lpvs_window_count(len(t), n, nov))
    S = np.zeros((len(f), 3, 3), dtype=np.complex128)
    Yc = np.ascontiguousarray(Y.T)
    N = len(t)

    def call(Cn=3, ldY=N, mu=0.05, pk=L.PROX_L1, k0=0, k1=K, Yh=Yc):
        return mctx.lib.lpvs_ls_window_matrix_sparse_sums(mctx.h, vp(Yh), Cn, ldY, vp(t), N, vp(f), len(f), vp(W), n, nov,
                                                          pk, 0.1, mu, 100, 1e-8, k0, k1, vp(S), None, None, None)

    assert call() == L.OK
    assert call(Cn=0) == L.E_BAD_ARG
    assert call(ldY=N - 1) == L.E_BAD_ARG
    assert call(mu=0.0) == L.E_BAD_ARG and call(mu=1.5) == L.E_BAD_ARG
    assert call(pk=L.PROX_GROUP_L2) == L.E_BAD_ARG and call(pk=-1) == L.E_BAD_ARG
    assert call(k0=-1) == L.E_BAD_ARG and call(k1=K + 1) == L.E_BAD_ARG and call(k0=2, k1=1) == L.E_BAD_ARG
    Yn = Yc.copy()
    Yn[1, 7] = np.nan
    assert call(Yh=Yn) == L.E_NONFINITE
    assert call() == L.OK  # the context stays usable
    for bad in (dict(init=True), dict(cb=lambda *a: None), dict(verbose=True, printerval=10, iters=100)):
        with pytest.raises(TypeError):
            lp.ls_sparse_windowcsd_matrix(Y, t, f, ctx=mctx, **bad)
    with pytest.raises(TypeError):
        lp.ls_sparse_cohere_matrix(Y, t, f, window_func=lp.rect, ctx=mctx)
    # float32 in: float32 / complex64 out, the FP64 answer rounded
    kw = dict(nw=3, noverlap=nov, window_func=lp.hanning, iters=500, tol=1e-9, ctx=mctx)
    Y32 = Y.astype(np.float32)
    S32, _ = lp.ls_sparse_windowcsd_matrix(Y32, t, f, **kw)
    S64, _ = lp.ls_sparse_windowcsd_matrix(Y32.astype(np.float64), t, f, **kw)
    assert S32.dtype == np.complex64 and np.array_equal(S32, S64.astype(np.complex64))
    P32, _ = lp.ls_sparse_windowpsd_multi(Y32, t, f, **kw)
    assert P32.dtype == np.float32


def test_verbose(mctx, capsys):
    import lpvspectral_jl_b200 as lp

    t, Y = record(3 * 101, 2, 6)
    f = np.arange(1, 9) * 0.5 / (t[101] - t[0])
    lp.ls_sparse_windowpsd_multi(Y, t, f, nw=3, noverlap=50, verbose=True, iters=2000, tol=1e-6, ctx=mctx)
    lines = capsys.readouterr().out.strip().splitlines()
    assert len(lines) == mctx.last_window_iters.size and all("||x-z||₂" in ln for ln in lines)
