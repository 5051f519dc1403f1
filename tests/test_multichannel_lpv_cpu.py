"""ls_spectral_lpv_multi / ls_windowpsd_lpv_multi without a GPU: the channel layout and defaults handed to the C ABI (through
a stand-in context that records the call), the list of SpectralExt with Σ = var_e[c] * Sigma0, the per-channel warnings,
eltypes, validation before any device call, and the new symbols' presence in the header, the bindings and the library.
CPU only."""
import ctypes as C
import os
import re
import warnings

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NF, NV = 3, 2


def _arr(p, n):
    return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(n,))


class _FakeLib:
    def __init__(self, fva=(0.95, 0.5, 0.99)):
        self.calls = []
        self.fva = fva

    def lpvs_ls_spectral_lpv_multi(self, h, Y, nch, ldY, X, V, N, w, Nf, Nv, lam, coulomb, normalize, params, Sigma0,
                                   var_e, fva, info):
        self.calls.append(dict(Y=_arr(Y, nch * ldY).copy(), C=nch, ldY=ldY, N=N, Nf=Nf, Nv=Nv, lam=lam,
                               coulomb=coulomb, normalize=normalize, Sigma0=Sigma0))
        ncc = Nf * Nv * (2 if coulomb else 1)
        _arr(params, 2 * ncc * nch)[:] = np.arange(2 * ncc * nch)  # channel c's ncc complex values at 2 c ncc
        if Sigma0 is not None:
            _arr(Sigma0, 4 * ncc * ncc)[:] = np.arange(4 * ncc * ncc) + 1.0
        _arr(var_e, nch)[:] = np.arange(nch) + 2.0
        _arr(fva, nch)[:] = self.fva[:nch]
        for c in range(nch):
            info[c] = c
        return 0

    def lpvs_ls_windowpsd_lpv_multi(self, h, Y, nch, ldY, X, V, N, w, Nf, Nv, n, noverlap, lam, coulomb, normalize, S,
                                    fva, K, info):
        self.calls.append(dict(C=nch, ldY=ldY, N=N, Nf=Nf, n=n, noverlap=noverlap, lam=lam))
        _arr(S, Nf * nch)[:] = np.arange(Nf * nch)  # channel c at S + c Nf
        K._obj.value = 2
        f = _arr(fva, 2 * nch)
        f[:] = 1.0
        f[nch + 1] = 0.3  # window 1, channel 1
        return 0


class _FakeCtx:
    h = None

    def __init__(self, **kw):
        self.lib = _FakeLib(**kw)

    def check(self, rc):
        assert rc == 0


def _inputs(N=40, nch=3):
    rng = np.random.default_rng(0)
    return rng.standard_normal((N, nch)), rng.random(N), rng.random(N), 2 * np.pi * np.arange(1, NF + 1, dtype=float)


def test_layout_defaults_and_sigma(monkeypatch):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _api

    Y, X, V, w = _inputs()
    seen = []
    orig = _api._channels
    monkeypatch.setattr(_api, "_channels", lambda a: seen.append(a) or orig(a))
    ctx = _FakeCtx()
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        out, info = lp.ls_spectral_lpv_multi(Y, X, V, w, NV, ctx=ctx, return_info=True)
    assert len(seen) == 1  # the channel layout of the other multi-channel estimators
    call = ctx.lib.calls[0]
    assert call["C"] == 3 and call["ldY"] == 40 and call["N"] == 40 and call["lam"] == 1e-8
    assert call["Nf"] == NF and call["Nv"] == NV and call["coulomb"] == 0 and call["normalize"] == 1
    assert np.array_equal(call["Y"], np.ascontiguousarray(Y.T).ravel())
    assert isinstance(out, list) and len(out) == 3 and all(isinstance(se, lp.SpectralExt) for se in out)
    ncc = NF * NV
    S0 = (np.arange(4 * ncc * ncc) + 1.0).reshape(2 * ncc, 2 * ncc)
    for c, se in enumerate(out):
        assert np.array_equal(se.Y, Y[:, c])
        assert se.x.dtype == np.complex128 and se.x.shape == (ncc,)
        assert se.x[1] == complex(2 * c * ncc + 2, 2 * c * ncc + 3)  # channel c at 2 c ncc doubles
        assert np.array_equal(se.Σ, (c + 2.0) * S0)  # var_e[c] * Sigma0
        assert se.fva == [0.95, 0.5, 0.99][c] and se.λ == 1e-8 and se.Nv == NV
    assert list(info) == [0, 1, 2]
    msgs = [str(r.message) for r in rec]
    assert msgs == ["Fraction of variance explained = 0.5"]  # once, for the one channel under 0.9
    out2 = lp.ls_spectral_lpv_multi(Y, X, V, w, NV, λ=0.02, coulomb=True, normalize=False, want_sigma=False, ctx=ctx)
    call = ctx.lib.calls[-1]
    assert call["lam"] == 0.02 and call["coulomb"] == 1 and call["normalize"] == 0 and call["Sigma0"] is None
    assert all(se.Σ is None for se in out2) and out2[0].x.shape == (2 * ncc,)
    one = lp.ls_spectral_lpv_multi(Y[:, 0], X, V, w, NV, lam=1e-3, ctx=_FakeCtx())  # a 1-D signal is one channel
    assert len(one) == 1


def test_windowed_layout_and_warnings():
    import lpvspectral_jl_b200 as lp

    Y, X, V, w = _inputs()
    ctx = _FakeCtx()
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        S = lp.ls_windowpsd_lpv_multi(Y, X, V, w, NV, ctx=ctx)
    call = ctx.lib.calls[0]
    assert call["C"] == 3 and call["ldY"] == 40 and call["n"] == 4 and call["noverlap"] == 0 and call["lam"] == 1e-8
    assert S.shape == (NF, 3) and S[1, 2] == 2 * NF + 1  # column c = channel c
    assert [str(r.message) for r in rec] == ["Fraction of variance explained = 0.3"]  # per (window, channel)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        lp.ls_windowpsd_lpv_multi(Y, X, V, w, NV, 4, 5, λ=0.1, ctx=ctx)
    assert ctx.lib.calls[-1]["n"] == 10 and ctx.lib.calls[-1]["noverlap"] == 5 and ctx.lib.calls[-1]["lam"] == 0.1


def test_float32_gives_complex64():
    import lpvspectral_jl_b200 as lp

    Y, X, V, w = _inputs()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out, _ = lp.ls_spectral_lpv_multi(Y.astype(np.float32), X, V, w, NV, ctx=_FakeCtx(), return_info=True)
        S = lp.ls_windowpsd_lpv_multi(Y.astype(np.float32), X, V, w, NV, ctx=_FakeCtx())
    assert all(se.x.dtype == np.complex64 and se.Σ.dtype == np.float32 for se in out)
    assert S.dtype == np.float32


def test_argument_validation():
    import lpvspectral_jl_b200 as lp

    Y, X, V, w = _inputs()
    ctx = _FakeCtx()
    for fn in (lp.ls_spectral_lpv_multi, lp.ls_windowpsd_lpv_multi):
        with pytest.raises(ValueError):
            fn(Y, X[:-1], V, w, NV, ctx=ctx)
        with pytest.raises(ValueError):
            fn(Y, X, V[:-1], w, NV, ctx=ctx)
        with pytest.raises(ValueError):
            fn(np.zeros((40, 0)), X, V, w, NV, ctx=ctx)
        with pytest.raises(ValueError):
            fn(np.zeros((40, 2, 2)), X, V, w, NV, ctx=ctx)
        with pytest.raises(TypeError):
            fn(Y, X, V, w, NV, ctx=ctx, iters=3)
    assert ctx.lib.calls == []


def test_symbols_are_declared_bound_and_exported():
    from lpvspectral_jl_b200 import _lib as L

    syms = L.declared_symbols()
    shim = open(os.path.join(ROOT, "julia", "LPVSpectralB200.jl")).read()
    exported = re.search(r"export ([^\n]*\n(?:\s+[^\n]*\n)*)", shim).group(1)
    for s in ("lpvs_ls_spectral_lpv_multi", "lpvs_ls_windowpsd_lpv_multi"):
        assert s in syms and s in L._PROTOS
        assert hasattr(L.load(), s)
        assert f"(:{s}, liblpvs)" in shim
    for name in ("ls_spectral_lpv_multi", "ls_windowpsd_lpv_multi"):
        assert re.search(rf"\b{name}\b", exported)
