"""ls_spectral_multi without a GPU: argument validation, shapes and eltypes, the channel layout handed to the C ABI (through a
stand-in context that records the call), and the new symbols' presence in the library's exports.  CPU only."""
import ctypes as C

import numpy as np
import pytest


class _FakeLib:
    def __init__(self):
        self.calls = []

    def lpvs_ls_spectral_multi(self, h, Y, nch, ldY, t, N, f, Nf, W, lam, X, info):
        self.calls.append(dict(Y=Y.value, C=nch, ldY=ldY, N=N, Nf=Nf, W=W, lam=lam))
        x = np.ctypeslib.as_array(C.cast(X, C.POINTER(C.c_double)), shape=(2 * nch * Nf,))
        x[:] = np.arange(2 * nch * Nf)  # channel c's Nf complex values at 2 c Nf
        info[0] = 3
        return 0


class _FakeCtx:
    h = None

    def __init__(self):
        self.lib = _FakeLib()

    def check(self, rc):
        assert rc == 0


def _inputs(N=50, nch=3):
    rng = np.random.default_rng(0)
    return rng.standard_normal((N, nch)), np.sort(rng.random(N))


def test_shapes_defaults_and_channel_layout(monkeypatch):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _api

    Y, t = _inputs()
    seen = []
    orig = _api._channels
    monkeypatch.setattr(_api, "_channels", lambda a: seen.append(a) or orig(a))
    ctx = _FakeCtx()
    X, f, info = lp.ls_spectral_multi(Y, t, ctx=ctx, return_info=True)
    assert len(seen) == 1  # the channel layout of the matrix estimators, not a copy of it
    call = ctx.lib.calls[0]
    assert call["C"] == 3 and call["ldY"] == 50 and call["N"] == 50 and call["W"] is None and call["lam"] == 1e-10
    assert np.array_equal(f, lp.default_freqs(t)) and call["Nf"] == len(f)
    assert X.shape == (len(f), 3) and X.dtype == np.complex128
    Nf = len(f)
    assert X[1, 2] == complex(2 * (2 * Nf + 1), 2 * (2 * Nf + 1) + 1)  # column c = channel c, fourier2complex order
    assert info.shape == (3,) and info[0] == 3
    X2, f2 = lp.ls_spectral_multi(Y, t, [0.0, 1.0, 2.0], np.ones(50), λ=1e-3, ctx=ctx)
    assert X2.shape == (3, 3) and ctx.lib.calls[-1]["lam"] == 1e-3 and ctx.lib.calls[-1]["W"] is not None
    X1, _ = lp.ls_spectral_multi(Y[:, 0], t, ctx=ctx)  # a 1-D signal is one channel
    assert X1.shape == (len(f), 1)


def test_float32_gives_complex64():
    import lpvspectral_jl_b200 as lp

    Y, t = _inputs()
    X, _ = lp.ls_spectral_multi(Y.astype(np.float32), t, ctx=_FakeCtx())
    assert X.dtype == np.complex64


def test_argument_validation():
    import lpvspectral_jl_b200 as lp

    Y, t = _inputs()
    ctx = _FakeCtx()
    with pytest.raises(ValueError):
        lp.ls_spectral_multi(Y, t[:-1], ctx=ctx)
    with pytest.raises(ValueError):
        lp.ls_spectral_multi(Y, t, None, np.ones(49), ctx=ctx)
    with pytest.raises(ValueError):
        lp.ls_spectral_multi(np.zeros((50, 0)), t, ctx=ctx)
    with pytest.raises(ValueError):
        lp.ls_spectral_multi(np.zeros((50, 2, 2)), t, ctx=ctx)
    with pytest.raises(TypeError):
        lp.ls_spectral_multi(Y, t, ctx=ctx, nw=3)
    with pytest.raises(Exception):
        lp.ls_spectral_multi(Y, t, [1.0, 0.0], ctx=ctx)  # a zero frequency must come first (check_freq)
    assert ctx.lib.calls == []


def test_symbols_are_declared_and_exported():
    from lpvspectral_jl_b200 import _lib as L

    syms = L.declared_symbols()
    for s in ("lpvs_ls_spectral_multi", "lpvs_ls_spectral_multi_dev"):
        assert s in syms
        assert hasattr(L.load(), s)
