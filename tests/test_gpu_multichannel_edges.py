"""GPU: the cross-spectral matrix path (lpvs_ls_window_matrix_sums[_dev]) at its channel, block and batch edges.

The reference is the literal oracle of tests/oracle_matrix.py: one N-rhs LU per window at the reference's phase rounding.
Channel c of every record is scaled by 10^((c mod 7) - 3), and each entry is checked against its own scale,
e_ij = |S_ij - R_ij|_2 / sqrt(|R_ii|_2 |R_jj|_2) <= max(1e-12, 40 cond eps), so a wrong quiet channel cannot hide in the norm
of a loud one.  The chunk classes of the kernels (csrc/chol.cu trsm_multi_chunk, csrc/gram.cu RHS_MC):
    k_trsm_multi<8>  for C <= 8,  k_trsm_multi<16> for 9 <= C <= 16,  k_trsm_multi<32> for C >= 17 (several CTAs for C > 32),
    k_gram_rhs_multi 4 channels per CTA,
so C in {8, 9, 16, 17, 32, 33, 65} runs every class with full and partial last chunks.  Nf in {64, 65, 129} gives
nb = Np / 128 = 1, 2, 3.  -m gpu."""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle import lpvs_oracle as o

import oracle_matrix as om
from test_gpu_multichannel import EPS, _dev_sums, _jitter_cond, bar, max_cond, record

pytestmark = pytest.mark.gpu

MODES = {"auto": 0, "chain": 1, "direct": 2, "chain_ref": 3, "structured": 4, "structured_ref": 5}


def scaled_record(N, nch, seed, T=10.0):
    """record(): every channel its own tone plus white noise (no S_ii(f) near 0), channel c scaled by 10^((c mod 7) - 3)."""
    t, Y = record(N, nch, seed, T)
    return t, Y * 10.0 ** ((np.arange(nch) % 7) - 3.0)


def entry_err(S, R):
    """(C, C) matrix of e_ij = |S_ij - R_ij|_2 / sqrt(|R_ii|_2 |R_jj|_2), the 2-norms over frequency."""
    d = np.sqrt(np.linalg.norm(np.einsum("fii->fi", R), axis=0))
    return np.linalg.norm(S - R, axis=0) / np.outer(d, d)


def grid(Nf, f0zero, Tw, nonuniform=False):
    if nonuniform:
        f = np.cumsum(1.0 + 0.5 * np.random.default_rng(Nf).random(Nf)) * 2.0 / Tw
        return np.concatenate([[0.0], f[:-1]]) if f0zero else f
    return (np.arange(Nf) + (0 if f0zero else 1)) * 2.0 / Tw


# name: (C, Nf, zero first frequency, n, nw, noverlap, non-uniform grid).  n is never a multiple of 32; N = nw n + nw - 1.
SHAPES = {
    "c8_nf65_f0zero": (8, 65, True, 417, 4, "half", False),
    "c9_nf129": (9, 129, False, 833, 3, "zero", False),
    "c9_nf64_f0zero": (9, 64, True, 389, 3, "half", False),
    "c17_nf16_hop1": (17, 16, False, 97, 2, "n-1", False),
    "c16_nf65": (16, 65, False, 431, 4, "half", False),
    "c17_nf129_f0zero": (17, 129, True, 811, 3, "half", False),
    "c17_nf1_n29": (17, 1, False, 29, 5, "half", False),
    "c32_nf65_f0zero": (32, 65, True, 419, 3, "zero", False),
    "c33_nf65": (33, 65, False, 427, 4, "half", False),
    "c33_nf64": (33, 64, False, 397, 3, "half", False),
    "c65_nf129_f0zero": (65, 129, True, 805, 3, "zero", False),
    "c9_nf65_f0zero_nonuniform": (9, 65, True, 417, 4, "half", True),
    "c33_nf65_nonuniform": (33, 65, False, 427, 3, "zero", True),
}
SHAPE_PARAMS = [(s, m) for s in SHAPES for m in (("auto", "direct") if SHAPES[s][6] else ("auto", "direct", "chain_ref"))]


@functools.lru_cache(maxsize=None)
def shape_case(name):
    nch, Nf, f0zero, n, nw, nov, nonuni = SHAPES[name]
    N = nw * n + nw - 1
    t, Y = scaled_record(N, nch, seed=N + nch)
    noverlap = {"half": n >> 1, "zero": 0, "n-1": n - 1}[nov]
    f = grid(Nf, f0zero, t[n] - t[0], nonuni)
    Sr, _ = om.ls_windowcsd_matrix(Y, t, f, nw=nw, noverlap=noverlap, window_func=o.hanning)
    Cr, _ = om.ls_cohere_matrix(Y, t, f, nw=nw, noverlap=noverlap)
    Pr, _ = om.ls_windowpsd_multi(Y, t, f, nw=nw, noverlap=noverlap, window_func=o.hanning)
    return t, Y, f, nw, noverlap, Sr, Cr, Pr, bar(max_cond(t, f, n, noverlap, o.hanning(n)))


@pytest.mark.parametrize("shape,mode", SHAPE_PARAMS)
def test_shapes_against_literal_oracle(ctx, shape, mode):
    """Every entry, coherence and PSD column against the oracle.  All (i, j) are checked at every C: the oracle has them all."""
    import lpvspectral_jl_b200 as lp

    t, Y, f, nw, noverlap, Sr, Cr, Pr, tol = shape_case(shape)
    with ctx.phase_mode(MODES[mode]):
        S, _ = lp.ls_windowcsd_matrix(Y, t, f, nw=nw, noverlap=noverlap, window_func=lp.hanning, ctx=ctx)
        Co, _ = lp.ls_cohere_matrix(Y, t, f, nw=nw, noverlap=noverlap, ctx=ctx)
        P, _ = lp.ls_windowpsd_multi(Y, t, f, nw=nw, noverlap=noverlap, window_func=lp.hanning, ctx=ctx)
    e = entry_err(S, Sr)
    i, j = np.unravel_index(np.argmax(e), e.shape)
    assert e.max() <= tol, (f"worst entry ({i}, {j})", e.max(), tol)
    ec = np.abs(Co - Cr).max(axis=0)
    i, j = np.unravel_index(np.argmax(ec), ec.shape)
    assert ec.max() <= 4 * tol, (f"worst coherence ({i}, {j})", ec.max(), 4 * tol)
    ep = np.linalg.norm(P - Pr, axis=0) / np.linalg.norm(Pr, axis=0)
    assert ep.max() <= tol, (f"worst PSD column {np.argmax(ep)}", ep.max(), tol)


# ---- exact properties: each channel's arithmetic depends neither on the chunk that holds it nor on C -------------------------
EXACT_PARAMS = [("uniform", m) for m in MODES] + [("nonuniform", m) for m in ("auto", "direct")]


@functools.lru_cache(maxsize=None)
def exact_case(grid_kind):
    """C = 33 (k_trsm_multi<32>: a full chunk and one of 1 channel), Nf = 129 (nb = 3), t over [0, 20]: the batches of 3 of
    the 7 windows reach max|t| of about 10, 17.5 and 20, and a batch of 1 about 5 -- different binades."""
    n, nch = 811, 33
    N = n + 6 * (n - (n >> 1))
    t, Y = scaled_record(N, nch, seed=77, T=20.0)
    f = grid(129, False, t[n] - t[0], grid_kind == "nonuniform")
    return t, Y, f, o.hanning(n), n, n >> 1


@pytest.mark.parametrize("grid_kind,mode", EXACT_PARAMS)
def test_exact_channel_properties(ctx, grid_kind, mode):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    t, Y, f, W, n, nov = exact_case(grid_kind)
    nch = Y.shape[1]
    K = lp.window_count(len(t), n, nov)
    assert K == 7

    def sums(Ym, k0=0, k1=K):
        return lp.window_matrix_sums(Ym, t, f, W, n, nov, 1e-10, k0, k1, ctx=ctx)

    with ctx.phase_mode(MODES[mode]):
        full = sums(Y)
        # a pair on its own gives the bits of the pair inside the C = 33 call (pairs straddle 4- and 32-channel chunks)
        for i, j in [(3, 4), (7, 8), (31, 32), (0, 32), (32, 15), (16, 17)]:
            two = sums(Y[:, [i, j]])
            assert np.array_equal(two[:, 0, 1], full[:, i, j]), (i, j)
            assert np.array_equal(two[:, 0, 0], full[:, i, i]) and np.array_equal(two[:, 1, 1], full[:, j, j]), (i, j)
        # permuting the channels permutes S
        p = np.random.default_rng(5).permutation(nch)
        assert np.array_equal(sums(Y[:, p]), full[:, p][:, :, p])
        # channel 20 a copy of channel 5, channel 9 all zero; every other entry keeps its bits
        Y2 = Y.copy()
        Y2[:, 20] = Y2[:, 5]
        Y2[:, 9] = 0.0
        S2 = sums(Y2)
        assert np.array_equal(S2[:, 5, 20], S2[:, 5, 5]) and np.array_equal(S2[:, 20, 5], S2[:, 5, 5])
        Co = lp.window_matrix_finalize(L.WIN_COHERE, S2, K)
        assert np.all(Co[:, 5, 20] == 1.0) and np.all(Co[:, 20, 5] == 1.0)
        assert not S2[:, 9, :].any() and not S2[:, :, 9].any()
        keep = np.setdiff1d(np.arange(nch), [9, 20])
        assert np.array_equal(S2[:, keep][:, :, keep], full[:, keep][:, :, keep])
        # the factorisation batch does not change a bit, here and in the two-channel path
        pair = lp.window_sums(L.WIN_COHERE, Y[:, 0], Y[:, 32], t, f, W, n, nov, 1e-10, 0, K, ctx=ctx)
        for batch in (1, 3):
            ctx.set_option(L.OPT_WINDOW_BATCH, batch)
            try:
                Sb = sums(Y)
                pb = lp.window_sums(L.WIN_COHERE, Y[:, 0], Y[:, 32], t, f, W, n, nov, 1e-10, 0, K, ctx=ctx)
            finally:
                ctx.set_option(L.OPT_WINDOW_BATCH, 0)
            assert np.array_equal(Sb, full), batch
            assert np.array_equal(pb, pair), batch
        # host form against the device form, both from window 2, the device buffer with ldY > N
        assert np.array_equal(_dev_sums(ctx, Y, t, f, W, n, nov, 1e-10, 2, K, ldY=len(t) + 37), sums(Y, 2, K))


# ---- the per-window jitter retry and LPVS_E_NOT_SPD away from window 0 --------------------------------------------------------


@pytest.mark.parametrize("mode", ["auto", "structured_ref"])
def test_jitter_retry_in_later_batches_and_chunks(ctx, mode):
    """lam = -10 breaks down the factorisation of every window, so each is re-done alone with max(lam, Nreg eps max diag G).
    C = 33 (two trsm chunks), batches of 3 over windows [2, 12) (10 windows: the last batch holds one)."""
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    n, nch, K, k0 = 500, 33, 12, 2
    t, Y = scaled_record(K * n, nch, seed=19)
    f = np.arange(64) * 2.0 / (t[n] - t[0])
    W = o.hanning(n)
    Yc = np.ascontiguousarray(Y.T)
    sums = np.zeros((len(f), nch, nch), dtype=np.complex128)
    info = C.c_int(0)
    ctx.set_option(L.OPT_WINDOW_BATCH, 3)
    try:
        with ctx.phase_mode(MODES[mode]):
            ctx.check(ctx.lib.lpvs_ls_window_matrix_sums(ctx.h, Yc.ctypes.data_as(C.c_void_p), nch, K * n,
                                                         t.ctypes.data_as(C.c_void_p), K * n, f.ctypes.data_as(C.c_void_p),
                                                         len(f), W.ctypes.data_as(C.c_void_p), n, 0, -10.0, k0, K,
                                                         sums.ctypes.data_as(C.c_void_p), C.byref(info)))
    finally:
        ctx.set_option(L.OPT_WINDOW_BATCH, 0)
    assert info.value == L.INFO_JITTER
    ts, Ys = t[k0 * n:], Y[k0 * n:]
    ref, Kr, _ = om.matrix_sums(Ys, ts, f, nw=K - k0, noverlap=0, window_func=o.hanning, lam=-10.0, jitter=True)
    assert Kr == K - k0
    tol = bar(_jitter_cond(ts, f, n, W, lam=-10.0))
    assert tol < 1e-9
    e = entry_err(sums, ref)
    i, j = np.unravel_index(np.argmax(e), e.shape)
    assert e.max() <= tol, (f"worst entry ({i}, {j})", e.max(), tol)


def test_not_spd_names_the_absolute_window(ctx):
    """LPVS_OPT_JITTER = 0 and lam = 0: window 6 sits at t = 0 (f0 = 0: its -sin block is zero, the factorisation breaks
    down).  Called for windows [2, 10) in batches of 3, window 6 is in the second batch; every form names window 6."""
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    n, nch, K, bad = 400, 9, 10, 6
    t, Y = scaled_record(K * n, nch, seed=23)
    f = np.arange(48) * 2.0 / (t[n] - t[0])
    t[bad * n:(bad + 1) * n] = 0.0
    W = o.hanning(n)
    ctx.set_option(L.OPT_WINDOW_BATCH, 3)
    ctx.set_option(L.OPT_JITTER, 0)
    try:
        calls = {
            "matrix host": lambda: lp.window_matrix_sums(Y, t, f, W, n, 0, 0.0, 2, K, ctx=ctx),
            "matrix dev": lambda: _dev_sums(ctx, Y, t, f, W, n, 0, 0.0, 2, K, ldY=K * n + 3),
            "two-channel host": lambda: lp.window_sums(L.WIN_CSD, Y[:, 0], Y[:, 1], t, f, W, n, 0, 0.0, 2, K, ctx=ctx),
        }
        for form, call in calls.items():
            with pytest.raises(L.NotPositiveDefinite) as ei:
                call()
            assert f"window {bad} " in str(ei.value), (form, str(ei.value))
    finally:
        ctx.set_option(L.OPT_JITTER, 1)
        ctx.set_option(L.OPT_WINDOW_BATCH, 0)


# ---- LPVS_PHASE_STRUCTURED_REF on the matrix path at large phases -------------------------------------------------------------


def test_structured_ref_matrix_at_large_phases(ctx):
    """The setting of test_structured_ref_reproduces_reference_phase_rounding: t = 9.99 + 2.4e-3 U, phases up to 2.5e7 rad,
    where the reference's fl(fl(2 pi f) t) is off the ideal phase by up to ~3e-9 rad.  8 windows' worth (nw = 8, 15 windows with
    the default overlap), a uniform grid with cond(A'WA) ~ 1e3, C = 9.  The modes that take the reference's rounding match the
    oracle; the exact-phase modes (chain, structured) miss it by far more, so the correction is on this path.  Measured on a
    B200: worst entry error / bar 1.5e-5 (auto, direct, chain_ref), 1.5e-3 (structured_ref), 2.7 (chain) and 4.2 (structured),
    i.e. the exact-phase modes miss by about 1800x structured_ref's error."""
    import lpvspectral_jl_b200 as lp

    rng = np.random.default_rng(12)
    N, nw, nch = 4096, 8, 9
    t = 9.99 + np.sort(2.4e-3 * rng.random(N))
    _, Y = scaled_record(N, nch, seed=12)
    n = N // nw
    f = (np.arange(75) + 7) * 1.5 / (t[n] - t[0])
    cond = max_cond(t, f, n, n >> 1, o.hanning(n))
    tol = max(1e-9, 40.0 * cond * EPS)
    Sr, _ = om.ls_windowcsd_matrix(Y, t, f, nw=nw, window_func=o.hanning)
    err = {}
    for mode in MODES:
        with ctx.phase_mode(MODES[mode]):
            S, _ = lp.ls_windowcsd_matrix(Y, t, f, nw=nw, window_func=lp.hanning, ctx=ctx)
        err[mode] = entry_err(S, Sr).max()
    print(f"cond {cond:.2e}, bar {tol:.1e}; worst entry error / bar: "
          + ", ".join(f"{m} {e / tol:.2e}" for m, e in err.items()))
    for mode in ("auto", "direct", "chain_ref", "structured_ref"):
        assert err[mode] <= tol, (mode, err[mode], tol)
    for mode in ("chain", "structured"):
        assert err[mode] >= 100.0 * err["structured_ref"], (mode, err[mode], err["structured_ref"])
