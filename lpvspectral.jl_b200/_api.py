"""Host-side mirror of LPVSpectral.jl's least-squares estimators over the liblpvs C ABI.

Same names, argument meaning, defaults and error behaviour as the Julia functions (file:line into
/root/reference); all arithmetic happens in liblpvs.so on the GPU.  This module only marshals arguments
(collect ranges, evaluate ``window_func`` on the host, map ``proxg`` objects to (kind, param)) -- exactly what the
Julia shim in ``julia/LPVSpectralB200.jl`` does before its ``ccall``.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import math
import os
from dataclasses import dataclass
from typing import Callable, Optional

import numpy as np

from . import _lib as L

__all__ = [
    "Context", "default_context", "default_freqs", "check_freq", "rect", "hanning", "hamming", "window_count",
    "ls_spectral", "tls_spectral", "merge_windows", "mapwindows", "ls_windowpsd", "ls_windowcsd", "ls_cohere", "ls_spectral_lpv", "ls_sparse_spectral",
    "ls_sparse_spectral_lpv", "ls_windowpsd_lpv", "gram_fourier", "SpectralExt", "psd", "NormL1", "NormL0",
    "IndBallL0", "ADMM", "prox", "LpvsError", "NotPositiveDefinite", "window_sums", "window_sparse_sums", "window_finalize",
    "ls_windowpsd_multi", "ls_windowcsd_matrix", "ls_cohere_matrix", "window_matrix_sums", "window_matrix_finalize",
    "ls_sparse_windowpsd_multi", "ls_sparse_windowcsd_matrix", "ls_sparse_cohere_matrix", "window_matrix_sparse_sums",
    "ls_spectral_multi",
]

LpvsError = L.LpvsError
NotPositiveDefinite = L.NotPositiveDefinite


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel())


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _cast_like(val, single):
    if not single or not isinstance(val, np.ndarray):
        return val
    return val.astype(np.complex64 if np.iscomplexobj(val) else np.float32)


def _preserve_eltype(fn):
    """Float32 instantiation of the generic signatures (SURVEY 8f n2; e.g. src/lasso.jl:85 `AbstractArray{T}`): a
    Float32 signal gives Float32 / ComplexF32 results, as the reference's eltype-generic code does.  The dense solves run
    the library's FP64 path on the up-converted inputs; the sparse estimators additionally keep the ADMM inverse in single
    precision (half the bytes per iteration, double accumulation) -- either way at least as accurate as the reference's
    Float32 arithmetic."""
    import functools

    @functools.wraps(fn)
    def wrapper(y, *a, **k):
        single = isinstance(y, np.ndarray) and y.dtype == np.float32
        if single and fn.__name__ in ("ls_sparse_spectral", "ls_sparse_spectral_lpv"):
            k.setdefault("_m32", True)  # the ADMM loop streams the inverse in single precision (LPVS_OPT_ADMM_M32)
        out = fn(y, *a, **k)
        if not single:
            return out
        if isinstance(out, tuple):
            return (_cast_like(out[0], True),) + out[1:]
        if isinstance(out, SpectralExt):
            out.x = _cast_like(out.x, True)
            out.Σ = _cast_like(out.Σ, True)
            return out
        return _cast_like(out, True)

    return wrapper


PHASE_MODES = {"auto": L.PHASE_AUTO, "chain": L.PHASE_CHAIN, "direct": L.PHASE_DIRECT, "chain_ref": L.PHASE_CHAIN_REF,
               "structured": L.PHASE_STRUCTURED, "structured_ref": L.PHASE_STRUCTURED_REF}


class Context:
    """One liblpvs context = one GPU (one process per GPU)."""

    def __init__(self, device: Optional[int] = None):
        self.lib = L.load()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        h = C.c_void_p()
        rc = self.lib.lpvs_init(device, C.byref(h))
        if rc != L.OK:
            raise L.LpvsError(rc, f"lpvs_init(device={device}) failed: no usable B200 (there is no CPU fallback)")
        self.h = h
        self.device = device

    def check(self, rc):
        L.raise_for(rc, self.h)

    def set_option(self, key, value):
        self.check(self.lib.lpvs_set_option(self.h, key, float(value)))

    @contextlib.contextmanager
    def phase_mode(self, mode):
        """``with ctx.phase_mode("structured_ref"): ...`` -- LPVS_OPT_PHASE_MODE for the calls inside, then back to "auto".
        Names as in the Julia shim's ``phase_mode!``: auto, chain, direct, chain_ref, structured, structured_ref."""
        self.set_option(L.OPT_PHASE_MODE, PHASE_MODES[mode] if isinstance(mode, str) else int(mode))
        try:
            yield self
        finally:
            self.set_option(L.OPT_PHASE_MODE, L.PHASE_AUTO)

    def set_stream(self, cuda_stream_ptr):
        """Run on the caller's CUDA stream (e.g. ``torch.cuda.current_stream().cuda_stream``); 0/None = own stream."""
        self.check(self.lib.lpvs_set_stream(self.h, C.c_void_p(cuda_stream_ptr or 0)))

    @property
    def launches(self) -> int:
        return int(self.lib.lpvs_launch_count(self.h))

    def gram_timing(self):
        ms, n, fl = C.c_double(), C.c_int64(), C.c_double()
        self.lib.lpvs_last_gram_timing(self.h, C.byref(ms), C.byref(n), C.byref(fl))
        return ms.value, n.value, fl.value

    def last_call_ms(self) -> float:
        ms = C.c_double()
        self.check(self.lib.lpvs_last_call_ms(self.h, C.byref(ms)))
        return ms.value

    def release_workspace(self):
        """Give the grow-only device workspaces back (they are re-allocated on demand)."""
        self.check(self.lib.lpvs_release_workspace(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.lpvs_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default: Optional[Context] = None


def default_context() -> Context:
    global _default
    if _default is None:
        _default = Context()
    return _default


# ---- host-side helpers that stay host code in the reference too --------------------------------------------


def rect(n):
    return np.ones(int(n))


def hanning(n):
    n = int(n)
    if n == 1:
        return np.ones(1)
    return 0.5 * (1.0 - np.cos(2.0 * np.pi * np.arange(n) / (n - 1)))


def hamming(n):
    n = int(n)
    if n == 1:
        return np.ones(1)
    return 0.54 - 0.46 * np.cos(2.0 * np.pi * np.arange(n) / (n - 1))


def default_freqs(t, n: Optional[int] = None):
    """default_freqs(t) / default_freqs(t, n) (src/lsfft.jl:3-9)."""
    t = _f64(t)
    if n is not None:
        t = t[:n]
    fs = 1.0 / np.mean(np.diff(t))
    return np.arange(len(t) // 2 + 1, dtype=np.float64) * (fs / len(t))


def check_freq(f):
    """src/lsfft.jl:20-24: ArgumentError unless a zero frequency is first."""
    f = np.asarray(f)
    z = np.flatnonzero(f == 0)
    if len(z) and z[0] != 0:
        raise ValueError("If zero frequency is included it must be the first frequency")
    return 0 if len(z) else None


def window_count(N, n, noverlap=-1):
    return int(L.load().lpvs_window_count(int(N), int(n), int(noverlap)))


def _lam(kw, default):
    if "λ" in kw:
        return float(kw.pop("λ"))
    if "lam" in kw:
        return float(kw.pop("lam"))
    return default


# ---- estimators ---------------------------------------------------------------------------------------------


def gram_fourier(t, f, W=None, y=None, ctx: Optional[Context] = None):
    """A'WA (reference column order) and A'Wy from the fused synthesis kernel -- parity/bench entry."""
    ctx = ctx or default_context()
    t, f = _f64(t), _f64(f)
    Wv = None if W is None else _f64(W)
    yv = None if y is None else _f64(y)
    nreg = 2 * len(f) - (1 if f[0] == 0 else 0)
    G = np.empty((nreg, nreg))
    b = np.empty(nreg) if yv is not None else None
    ctx.check(ctx.lib.lpvs_gram_fourier(ctx.h, _ptr(yv), _ptr(t), len(t), _ptr(f), len(f), _ptr(Wv), _ptr(G),
                                        _ptr(b)))
    return (G, b) if yv is not None else G


@_preserve_eltype
def ls_spectral(y, t, f=None, W=None, *, verbose=False, ctx: Optional[Context] = None, return_info=False, **kw):
    """ls_spectral(y,t,f=default_freqs(t)[,W]; λ=1e-10) -> (x, f)   (src/lsfft.jl:62-80)."""
    lam = _lam(kw, 1e-10)
    if kw:
        raise TypeError(f"unexpected keyword arguments {sorted(kw)}")
    ctx = ctx or default_context()
    yv, tv = _f64(y), _f64(t)
    if len(yv) != len(tv):
        raise ValueError("y and t has to be the same length")
    f_in = default_freqs(tv) if f is None else f
    fv = _f64(f_in)
    check_freq(fv)
    Wv = None
    if W is not None:
        Wv = _f64(W)
        if len(Wv) != len(yv):
            raise ValueError("W and y has to be the same length")
    x = np.empty(len(fv), dtype=np.complex128)
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_spectral(ctx.h, _ptr(yv), _ptr(tv), len(yv), _ptr(fv), len(fv), _ptr(Wv), lam,
                                       _ptr(x), C.byref(info)))
    if return_info:
        return x, f_in, info.value
    return x, f_in


@_preserve_eltype
def tls_spectral(y, t, f=None, *, ctx: Optional[Context] = None, return_info=False):
    """tls_spectral(y,t,f=default_freqs(t)[1:end-1]) -> (x, f)   (src/lsfft.jl:87-99): total least squares."""
    ctx = ctx or default_context()
    yv, tv = _f64(y), _f64(t)
    if len(yv) != len(tv):
        raise ValueError("y and t has to be the same length")
    f_in = default_freqs(tv)[:-1] if f is None else f
    fv = _f64(f_in)
    check_freq(fv)
    x = np.empty(len(fv), dtype=np.complex128)
    its = C.c_int(0)
    ctx.check(ctx.lib.lpvs_tls_spectral(ctx.h, _ptr(yv), _ptr(tv), len(yv), _ptr(fv), len(fv), _ptr(x), C.byref(its)))
    if return_info:
        return x, f_in, its.value
    return x, f_in


def merge_windows(pieces, N, n, noverlap=-1, ctx: Optional[Context] = None):
    """Base.merge(yf, w::Windows2) (src/windows.jl:58-70): overlap-average re-assembly of per-window outputs on the device."""
    ctx = ctx or default_context()
    P = np.ascontiguousarray(np.asarray(pieces, dtype=np.float64))
    if P.ndim != 2 or (P.size and P.shape[1] != n):
        raise ValueError("pieces must be K arrays of n samples")  # the reference: DimensionMismatch in ym[inds] .+= yf[i]
    out = np.empty(int(N))
    ctx.check(ctx.lib.lpvs_merge_windows(ctx.h, _ptr(P), P.shape[0], int(n), int(noverlap), int(N), _ptr(out)))
    return out


def mapwindows(fn: Callable, y, t, n, noverlap=-1, window_func: Callable = rect, ctx: Optional[Context] = None):
    """mapwindows(f, y, t, n, noverlap, window_func) (src/windows.jl:50-56): apply ``fn(y_i, t_i) -> yhat_i`` (an arbitrary
    host closure, as in the reference) to every window of Windows2 and merge the outputs (device overlap-average)."""
    yv, tv = _f64(y), _f64(t)
    if len(yv) != len(tv):
        raise ValueError("y and t has to be the same length")  # src/windows.jl:31
    n = int(n)
    if noverlap < 0:
        noverlap = n >> 1
    K = window_count(len(yv), n, noverlap)
    if K < 0:
        raise ValueError("noverlap must be smaller than the window length n")
    hop = n - noverlap
    pieces = np.empty((K, n))
    for k in range(K):
        sl = slice(k * hop, k * hop + n)
        out = np.asarray(fn(yv[sl], tv[sl]), dtype=np.float64)
        if out.shape != (n,):
            raise ValueError("f must return an output of the window's length")
        pieces[k] = out
    return merge_windows(pieces, len(yv), n, noverlap, ctx=ctx)


def window_sums(kind, y, u, t, freqs, W, n, noverlap, lam, k_begin, k_end, ctx: Optional[Context] = None):
    """Raw cross-window sums for windows [k_begin,k_end) -- the unit of multi-GPU sharding."""
    ctx = ctx or default_context()
    yv, tv = _f64(y), _f64(t)
    uv = None if u is None else _f64(u)
    fv, Wv = _f64(freqs), _f64(W)
    slen = {L.WIN_PSD: 1, L.WIN_CSD: 2, L.WIN_COHERE: 4}[kind] * len(fv)
    sums = np.zeros(slen)
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_window_sums(ctx.h, kind, _ptr(yv), _ptr(uv), _ptr(tv), len(yv), _ptr(fv), len(fv),
                                          _ptr(Wv), int(n), int(noverlap), float(lam), int(k_begin), int(k_end),
                                          _ptr(sums), C.byref(info)))
    return sums


def window_sparse_sums(kind, y, u, t, freqs, W, n, noverlap, proxg, mu, iters, tol, k_begin, k_end,
                       ctx: Optional[Context] = None, return_info=False):
    """Raw cross-window sums of the windowed estimators with estimator = ls_sparse_spectral for windows
    [k_begin,k_end): every window an independent device ADMM (lpvs_ls_window_sparse_sums) -- the sharding unit."""
    ctx = ctx or default_context()
    yv, tv, fv, Wv = _f64(y), _f64(t), _f64(freqs), _f64(W)
    uv = None if u is None else _f64(u)
    pk, pp = _prox_desc(proxg)
    nrhs = 1 if kind == L.WIN_PSD else 2
    sums = np.zeros({L.WIN_PSD: 1, L.WIN_CSD: 2, L.WIN_COHERE: 4}[kind] * len(fv))
    nk = max(int(k_end) - int(k_begin), 1)
    its = np.zeros(nk * nrhs, dtype=np.int64)
    res = np.zeros(nk * nrhs)
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_window_sparse_sums(ctx.h, kind, _ptr(yv), _ptr(uv), _ptr(tv), len(yv), _ptr(fv), len(fv),
                                                 _ptr(Wv), int(n), int(noverlap), pk, pp, float(mu), int(iters),
                                                 float(tol), int(k_begin), int(k_end), _ptr(sums), _ptr(its),
                                                 _ptr(res), C.byref(info)))
    if return_info:
        return sums, its.reshape(nk, nrhs), res.reshape(nk, nrhs)
    return sums


def window_finalize(kind, sums, Nf, K):
    sums = _f64(sums)
    out = np.empty(Nf, dtype=np.complex128 if kind == L.WIN_CSD else np.float64)
    rc = L.load().lpvs_ls_window_finalize(kind, _ptr(sums), int(Nf), int(K), _ptr(out))
    if rc != L.OK:
        raise ValueError("bad arguments to lpvs_ls_window_finalize")
    return out


def _windowed(kind, y, u, t, freqs, nw, noverlap, window_func, estimator, ctx, kw):
    ctx = ctx or default_context()
    yv, tv = _f64(y), _f64(t)
    uv = None if u is None else _f64(u)
    if len(yv) != len(tv) or (uv is not None and len(uv) != len(tv)):
        raise ValueError("y, t and v has to be the same length")  # src/windows.jl:31,96
    n = len(yv) // int(nw)  # src/lsfft.jl:113
    if freqs is None:
        freqs = default_freqs(tv, n)  # first window only (Q6)
    fv = _f64(freqs)
    check_freq(fv)
    if noverlap < 0:
        noverlap = n >> 1
    Wv = _f64(window_func(n))
    if len(Wv) != n:  # the reference broadcasts W against an n-sample window: DimensionMismatch (src/lsfft.jl:77)
        raise ValueError(f"window_func(n) must return n = {n} weights, got {len(Wv)}")
    K = window_count(len(yv), n, noverlap)
    if K < 0:  # DSP.arraysplit: ArgumentError
        raise ValueError("noverlap must be smaller than the window length n")
    # K == 0 (signal shorter than one window): the reference divides empty sums by K^2 / K -> NaN spectra; so do
    # lpvs_ls_window / window_finalize (0/0), deliberately not an error
    if estimator is None or estimator is ls_spectral:
        lam = _lam(kw, 1e-10)
        if kw:
            raise TypeError(f"unexpected keyword arguments {sorted(kw)}")
        out = np.empty(len(fv), dtype=np.complex128 if kind == L.WIN_CSD else np.float64)
        Kc = C.c_int64(0)
        info = C.c_int(0)
        ctx.check(ctx.lib.lpvs_ls_window(ctx.h, kind, _ptr(yv), _ptr(uv), _ptr(tv), len(yv), _ptr(fv), len(fv),
                                         _ptr(Wv), n, int(noverlap), lam, _ptr(out), C.byref(Kc), C.byref(info)))
        return out, freqs
    if estimator is not ls_sparse_spectral:
        raise ValueError("estimator must be ls_spectral or ls_sparse_spectral (no host-side fallback)")
    # estimator = ls_sparse_spectral (src/lsfft.jl:121, test/test_lasso.jl:36)
    kws = dict(kw)
    verbose = bool(kws.get("verbose", False))
    batched = not kws.get("init", False) and kws.get("cb") is None and not (
        verbose and kws.get("printerval", 100) < kws.get("iters", 10000))
    if batched:
        # all windows in one device pass: batched Gram / Cholesky / inverse, one CTA per window runs its ADMM
        lam = _lam(kws, 1.0)
        for key in ("init", "cb", "verbose"):
            kws.pop(key, None)
        kws.pop("printerval", None)
        iters, tol = int(kws.pop("iters", 10000)), float(kws.pop("tol", 1e-5))
        mu_kw = kws.pop("μ", kws.pop("mu", None))
        mu = 0.05 if mu_kw is None else float(mu_kw)
        proxg = kws.pop("proxg", None)
        if kws:
            raise TypeError(f"unexpected keyword arguments {sorted(kws)}")
        if not (0 <= mu <= 1):
            raise AssertionError("μ should be ≤ 1")  # src/lasso.jl:143
        pk, pp = _prox_desc(proxg if proxg is not None else NormL1(lam))
        nrhs = 1 if kind == L.WIN_PSD else 2
        sums = np.zeros({L.WIN_PSD: 1, L.WIN_CSD: 2, L.WIN_COHERE: 4}[kind] * len(fv))
        its = np.zeros(max(K, 1) * nrhs, dtype=np.int64)
        res = np.zeros(max(K, 1) * nrhs)
        info = C.c_int(0)
        if K > 0:
            ctx.check(ctx.lib.lpvs_ls_window_sparse_sums(ctx.h, kind, _ptr(yv), _ptr(uv), _ptr(tv), len(yv), _ptr(fv),
                                                         len(fv), _ptr(Wv), n, int(noverlap), pk, pp, mu, iters, tol,
                                                         0, K, _ptr(sums), _ptr(its), _ptr(res), C.byref(info)))
        if verbose:  # the line the reference prints when a window stops (src/lasso.jl:164-166)
            for k in range(K * nrhs):
                if res[k] < tol:
                    print("%d ||x-z||₂ %.10f" % (its[k], res[k]))
        ctx.last_window_iters = its[:K * nrhs].reshape(K, nrhs)
        return window_finalize(kind, sums, len(fv), K), freqs
    # init / callbacks / periodic prints: one device ADMM solve per window through the single-problem entry point
    hop = n - noverlap
    Nf = len(fv)
    Syy, Suu = np.zeros(Nf), np.zeros(Nf)
    Syu = np.zeros(Nf, dtype=np.complex128)
    for k in range(K):
        sl = slice(k * hop, k * hop + n)
        xy = ls_sparse_spectral(yv[sl], tv[sl], fv, Wv, ctx=ctx, **dict(kw))[0]
        Syy += xy.real * xy.real + xy.imag * xy.imag
        if uv is not None:
            xu = ls_sparse_spectral(uv[sl], tv[sl], fv, Wv, ctx=ctx, **dict(kw))[0]
            Suu += xu.real * xu.real + xu.imag * xu.imag
            Syu += (xy.real * xu.real + xy.imag * xu.imag) + 1j * (xy.imag * xu.real - xy.real * xu.imag)
    if kind == L.WIN_PSD:
        return Syy / float(K) ** 2, freqs
    if kind == L.WIN_CSD:
        return (Syu.real / K) + 1j * (Syu.imag / K), freqs
    return (Syu.real * Syu.real + Syu.imag * Syu.imag) / (Suu * Syy), freqs


@_preserve_eltype
def ls_windowpsd(y, t, freqs=None, *, nw=8, noverlap=-1, window_func: Callable = rect, estimator=None, ctx=None,
                 **kw):
    """ls_windowpsd (src/lsfft.jl:112-126): S = Σ|x_i|²/K², weighted estimator per window."""
    return _windowed(L.WIN_PSD, y, None, t, freqs, nw, noverlap, window_func, estimator, ctx, kw)


@_preserve_eltype
def ls_windowcsd(y, u, t, freqs=None, *, nw=10, noverlap=-1, window_func: Callable = rect, estimator=None,
                 ctx=None, **kw):
    """ls_windowcsd (src/lsfft.jl:140-156): S = Σ xy·conj(xu)/K."""
    return _windowed(L.WIN_CSD, y, u, t, freqs, nw, noverlap, window_func, estimator, ctx, kw)


@_preserve_eltype
def ls_cohere(y, u, t, freqs=None, *, nw=10, noverlap=-1, estimator=None, ctx=None, **kw):
    """ls_cohere (src/lsfft.jl:176-193): window hard-coded to hanning (Q8)."""
    if "window_func" in kw:
        raise TypeError("ls_cohere does not accept window_func (hanning is hard-coded, src/lsfft.jl:182)")
    return _windowed(L.WIN_COHERE, y, u, t, freqs, nw, noverlap, hanning, estimator, ctx, kw)


# ---- many channels at shared sample positions: one Gram matrix and one factor per window for all of them ----------------


def _channels(Y):
    """N x C (a 1-D signal is one channel) -> C x N contiguous float64: channel c at offset c N, i.e. ldY = N.

    A Fortran-ordered (column-major) float64 Y is used in place.  A C-ordered one has to be transposed on the host; that is
    done in blocks of rows that stay in cache (about 3x faster than one strided copy for N = 2^22, C = 32)."""
    Yv = np.asarray(Y, dtype=np.float64)
    if Yv.ndim == 1:
        Yv = Yv[:, None]
    if Yv.ndim != 2 or Yv.shape[1] < 1:
        raise ValueError("Y must be an N x C matrix with C >= 1")
    if Yv.T.flags.c_contiguous or Yv.shape[1] == 1:
        return np.ascontiguousarray(Yv.T)
    out = np.empty((Yv.shape[1], Yv.shape[0]))
    for r in range(0, Yv.shape[0], 1024):
        out[:, r:r + 1024] = Yv[r:r + 1024].T
    return out


@_preserve_eltype
def ls_spectral_multi(Y, t, f=None, W=None, *, ctx: Optional[Context] = None, return_info=False, **kw):
    """ls_spectral of every column of Y (N x C) at the shared sample positions t -> (X, f[, info]): X is (Nf, C) complex,
    column c what ls_spectral(Y[:, c], t, f, W; λ) computes (λ=1e-10), info (C,) the route flag of each channel.  The Gram
    matrix and its factors depend only on t, W and f, so they are built once for all channels (lpvs_ls_spectral_multi)."""
    lam = _lam(kw, 1e-10)
    if kw:
        raise TypeError(f"unexpected keyword arguments {sorted(kw)}")
    Yc, tv = _channels(Y), _f64(t)
    C_, N = Yc.shape
    if N != len(tv):
        raise ValueError("Y and t has to be the same length")
    f_in = default_freqs(tv) if f is None else f
    fv = _f64(f_in)
    check_freq(fv)
    Wv = None
    if W is not None:
        Wv = _f64(W)
        if len(Wv) != N:
            raise ValueError("W and Y has to be the same length")
    ctx = ctx or default_context()
    X = np.empty((C_, len(fv)), dtype=np.complex128)
    info = np.zeros(C_, dtype=np.int32)
    ctx.check(ctx.lib.lpvs_ls_spectral_multi(ctx.h, _ptr(Yc), C_, N, _ptr(tv), N, _ptr(fv), len(fv), _ptr(Wv), lam,
                                             _ptr(X), info.ctypes.data_as(C.POINTER(C.c_int))))
    if return_info:
        return X.T, f_in, info
    return X.T, f_in


def window_matrix_sums(Y, t, freqs, W, n, noverlap, lam, k_begin, k_end, ctx: Optional[Context] = None):
    """Raw cross-window sums of the C x C cross-spectral matrix for windows [k_begin,k_end) (lpvs_ls_window_matrix_sums):
    Y is N x C, returns an (Nf, C, C) complex array, entry [f, i, j] = sum_k x_i(f) conj(x_j(f)) -- the sharding unit."""
    ctx = ctx or default_context()
    Yc, tv, fv, Wv = _channels(Y), _f64(t), _f64(freqs), _f64(W)
    C_, N = Yc.shape
    sums = np.zeros((len(fv), C_, C_), dtype=np.complex128)
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_window_matrix_sums(ctx.h, _ptr(Yc), C_, N, _ptr(tv), N, _ptr(fv), len(fv), _ptr(Wv), int(n),
                                                 int(noverlap), float(lam), int(k_begin), int(k_end), _ptr(sums),
                                                 C.byref(info)))
    return sums


def window_matrix_finalize(kind, sums, K):
    """lpvs_ls_window_matrix_finalize: PSD (Nf, C) = S_cc / K^2, CSD (Nf, C, C) = S / K, COHERE (Nf, C, C) =
    abs2(S_ij) / (S_jj S_ii)."""
    S = np.ascontiguousarray(np.asarray(sums, dtype=np.complex128))
    Nf, C_ = S.shape[0], S.shape[1]
    shape = (Nf, C_) if kind == L.WIN_PSD else (Nf, C_, C_)
    out = np.empty(shape, dtype=np.complex128 if kind == L.WIN_CSD else np.float64)
    rc = L.load().lpvs_ls_window_matrix_finalize(kind, _ptr(S), int(Nf), int(C_), int(K), _ptr(out))
    if rc != L.OK:
        raise ValueError("bad arguments to lpvs_ls_window_matrix_finalize")
    return out


def _matrix_windows(Y, t, freqs, nw, noverlap, window_func):
    """Channels, window length, frequencies, weights and window count of the matrix estimators."""
    Yc, tv = _channels(Y), _f64(t)
    N = Yc.shape[1]
    if N != len(tv):
        raise ValueError("Y and t must have the same number of samples")
    n = N // int(nw)
    if freqs is None:
        freqs = default_freqs(tv, n)
    fv = _f64(freqs)
    check_freq(fv)
    if noverlap < 0:
        noverlap = n >> 1
    Wv = _f64(window_func(n))
    if len(Wv) != n:
        raise ValueError(f"window_func(n) must return n = {n} weights, got {len(Wv)}")
    K = window_count(N, n, noverlap)
    if K < 0:
        raise ValueError("noverlap must be smaller than the window length n")
    return Yc, tv, freqs, fv, Wv, n, noverlap, K


def _windowed_matrix(kind, Y, t, freqs, nw, noverlap, window_func, ctx, kw):
    lam = _lam(kw, 1e-10)
    if kw:  # the sparse estimator has its own names: ls_sparse_windowpsd_multi & co.
        raise TypeError(f"unexpected keyword arguments {sorted(kw)}")
    ctx = ctx or default_context()
    Yc, tv, freqs, fv, Wv, n, noverlap, K = _matrix_windows(Y, t, freqs, nw, noverlap, window_func)
    N = Yc.shape[1]
    sums = np.zeros((len(fv), Yc.shape[0], Yc.shape[0]), dtype=np.complex128)
    info = C.c_int(0)
    if K > 0:
        ctx.check(ctx.lib.lpvs_ls_window_matrix_sums(ctx.h, _ptr(Yc), Yc.shape[0], N, _ptr(tv), N, _ptr(fv), len(fv),
                                                     _ptr(Wv), n, int(noverlap), lam, 0, K, _ptr(sums), C.byref(info)))
    return window_matrix_finalize(kind, sums, K), freqs


@_preserve_eltype
def ls_windowpsd_multi(Y, t, freqs=None, *, nw=8, noverlap=-1, window_func: Callable = rect, ctx=None, **kw):
    """ls_windowpsd of every column of the N x C matrix Y (same t) -> (Nf x C, freqs); one factorisation per window."""
    return _windowed_matrix(L.WIN_PSD, Y, t, freqs, nw, noverlap, window_func, ctx, kw)


@_preserve_eltype
def ls_windowcsd_matrix(Y, t, freqs=None, *, nw=10, noverlap=-1, window_func: Callable = rect, ctx=None, **kw):
    """Cross-spectral matrix of the columns of Y (same t) -> (Nf x C x C complex, freqs); entry [:, i, j] is
    ls_windowcsd(Y[:, i], Y[:, j], t, ...)."""
    return _windowed_matrix(L.WIN_CSD, Y, t, freqs, nw, noverlap, window_func, ctx, kw)


@_preserve_eltype
def ls_cohere_matrix(Y, t, freqs=None, *, nw=10, noverlap=-1, ctx=None, **kw):
    """Coherence matrix of the columns of Y (same t) -> (Nf x C x C, freqs); entry [:, i, j] is ls_cohere(Y[:, i], Y[:, j],
    t, ...), the window hard-coded to hanning as there."""
    if "window_func" in kw:
        raise TypeError("ls_cohere_matrix does not accept window_func (hanning is hard-coded, as in ls_cohere)")
    return _windowed_matrix(L.WIN_COHERE, Y, t, freqs, nw, noverlap, hanning, ctx, kw)


# ---- many channels with estimator = ls_sparse_spectral: one inverse per window, each channel's ADMM once ------------


def window_matrix_sparse_sums(Y, t, freqs, W, n, noverlap, proxg, mu, iters, tol, k_begin, k_end,
                              ctx: Optional[Context] = None, return_info=False):
    """Raw cross-window sums of the sparse C x C cross-spectral matrix for windows [k_begin,k_end)
    (lpvs_ls_window_matrix_sparse_sums): Y is N x C, returns an (Nf, C, C) complex array, entry [f, i, j] =
    sum_k z_i(f) conj(z_j(f)); with return_info also the iteration counts and final residuals, (nwin, C) each."""
    ctx = ctx or default_context()
    Yc, tv, fv, Wv = _channels(Y), _f64(t), _f64(freqs), _f64(W)
    C_, N = Yc.shape
    pk, pp = _prox_desc(proxg)
    nk = max(int(k_end) - int(k_begin), 1)
    sums = np.zeros((len(fv), C_, C_), dtype=np.complex128)
    its = np.zeros((nk, C_), dtype=np.int64)
    res = np.zeros((nk, C_))
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_window_matrix_sparse_sums(ctx.h, _ptr(Yc), C_, N, _ptr(tv), N, _ptr(fv), len(fv), _ptr(Wv),
                                                        int(n), int(noverlap), pk, pp, float(mu), int(iters),
                                                        float(tol), int(k_begin), int(k_end), _ptr(sums), _ptr(its),
                                                        _ptr(res), C.byref(info)))
    if return_info:
        return sums, its, res
    return sums


def _sparse_matrix(kind, Y, t, freqs, nw, noverlap, window_func, ctx, kw):
    kws = dict(kw)
    for key in ("init", "cb"):
        if key in kws:
            raise TypeError(f"{key} is not offered by the matrix estimators (no per-window loop)")
    verbose = bool(kws.pop("verbose", False))
    iters, tol = int(kws.pop("iters", 10000)), float(kws.pop("tol", 1e-5))
    if "printerval" in kws and int(kws.pop("printerval")) < iters:
        raise TypeError("printerval < iters is not offered by the matrix estimators (no per-window loop)")
    lam = _lam(kws, 1.0)
    mu_kw = kws.pop("μ", kws.pop("mu", None))
    mu = 0.05 if mu_kw is None else float(mu_kw)
    proxg = kws.pop("proxg", None)
    if kws:
        raise TypeError(f"unexpected keyword arguments {sorted(kws)}")
    if not (0 <= mu <= 1):
        raise AssertionError("μ should be ≤ 1")  # src/lasso.jl:143
    proxg = proxg if proxg is not None else NormL1(lam)
    ctx = ctx or default_context()
    Yc, tv, freqs, fv, Wv, n, noverlap, K = _matrix_windows(Y, t, freqs, nw, noverlap, window_func)
    C_, N = Yc.shape
    sums = np.zeros((len(fv), C_, C_), dtype=np.complex128)
    its = np.zeros((K, C_), dtype=np.int64)
    res = np.zeros((K, C_))
    if K > 0:
        pk, pp = _prox_desc(proxg)
        info = C.c_int(0)
        ctx.check(ctx.lib.lpvs_ls_window_matrix_sparse_sums(ctx.h, _ptr(Yc), C_, N, _ptr(tv), N, _ptr(fv), len(fv),
                                                            _ptr(Wv), n, int(noverlap), pk, pp, mu, iters, tol, 0, K,
                                                            _ptr(sums), _ptr(its), _ptr(res), C.byref(info)))
    if verbose:  # the line the reference prints when a window stops (src/lasso.jl:164-166), per window and channel
        for k in range(K):
            for c in range(C_):
                if res[k, c] < tol:
                    print("%d ||x-z||₂ %.10f" % (its[k, c], res[k, c]))
    ctx.last_window_iters = its
    return window_matrix_finalize(kind, sums, K), freqs


@_preserve_eltype
def ls_sparse_windowpsd_multi(Y, t, freqs=None, *, nw=8, noverlap=-1, window_func: Callable = rect, ctx=None, **kw):
    """ls_windowpsd(..., estimator=ls_sparse_spectral) of every column of the N x C matrix Y (same t) -> (Nf x C, freqs).
    Keywords proxg (default NormL1(λ)), λ/lam = 1, μ/mu = 0.05, iters = 10000, tol = 1e-5, verbose; one inverse per
    window, each channel's ADMM once.  ctx.last_window_iters: (K, C) iteration counts."""
    return _sparse_matrix(L.WIN_PSD, Y, t, freqs, nw, noverlap, window_func, ctx, kw)


@_preserve_eltype
def ls_sparse_windowcsd_matrix(Y, t, freqs=None, *, nw=10, noverlap=-1, window_func: Callable = rect, ctx=None, **kw):
    """Sparse cross-spectral matrix of the columns of Y (same t) -> (Nf x C x C complex, freqs); entry [:, i, j] is
    ls_windowcsd(Y[:, i], Y[:, j], t, ..., estimator=ls_sparse_spectral).  Keywords as ls_sparse_windowpsd_multi."""
    return _sparse_matrix(L.WIN_CSD, Y, t, freqs, nw, noverlap, window_func, ctx, kw)


@_preserve_eltype
def ls_sparse_cohere_matrix(Y, t, freqs=None, *, nw=10, noverlap=-1, ctx=None, **kw):
    """Sparse coherence matrix of the columns of Y (same t) -> (Nf x C x C, freqs); entry [:, i, j] is
    ls_cohere(Y[:, i], Y[:, j], t, ..., estimator=ls_sparse_spectral), the window hard-coded to hanning as there."""
    if "window_func" in kw:
        raise TypeError("ls_sparse_cohere_matrix does not accept window_func (hanning is hard-coded, as in ls_cohere)")
    return _sparse_matrix(L.WIN_COHERE, Y, t, freqs, nw, noverlap, hanning, ctx, kw)


# ---- LPV --------------------------------------------------------------------------------------------------


@dataclass
class SpectralExt:
    """src/LPVSpectral.jl:59-70."""

    Y: np.ndarray
    X: np.ndarray
    V: np.ndarray
    w: np.ndarray
    Nv: int
    λ: float
    coulomb: bool
    normalize: bool
    x: np.ndarray
    Σ: Optional[np.ndarray]
    fva: Optional[float] = None


def psd(se: SpectralExt):
    """psd(se) (src/lsfft.jl:214-217): |Σ_k x[f,k]|²."""
    rp = np.reshape(se.x, (len(se.w), -1), order="F")
    s = rp.sum(axis=1)
    return s.real * s.real + s.imag * s.imag


@_preserve_eltype
def ls_spectral_lpv(Y, X, V, w, Nv, *, coulomb=False, normalize=True, want_sigma=True, ctx=None, **kw):
    """ls_spectral_lpv(Y,X,V,w,Nv; λ=1e-8, coulomb=false, normalize=true) -> SpectralExt (src/lsfft.jl:239-259)."""
    lam = _lam(kw, 1e-8)
    if kw:
        raise TypeError(f"unexpected keyword arguments {sorted(kw)}")
    ctx = ctx or default_context()
    Yv, Xv, Vv, wv = _f64(Y), _f64(X), _f64(V), _f64(w)
    if not (len(Yv) == len(Xv) == len(Vv)):
        raise ValueError("Y, X and V has to be the same length")
    nvv = (2 if coulomb else 1) * int(Nv)
    ncols = len(wv) * nvv
    params = np.empty(ncols, dtype=np.complex128)
    Sigma = np.empty((2 * ncols, 2 * ncols)) if want_sigma else None
    fva = C.c_double(0.0)
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_spectral_lpv(ctx.h, _ptr(Yv), _ptr(Xv), _ptr(Vv), len(Yv), _ptr(wv), len(wv), int(Nv),
                                           lam, int(bool(coulomb)), int(bool(normalize)), _ptr(params),
                                           _ptr(Sigma), C.byref(fva), C.byref(info)))
    if fva.value < 0.9:  # src/lsfft.jl:256
        import warnings

        warnings.warn(f"Fraction of variance explained = {fva.value}")
    return SpectralExt(Yv, Xv, Vv, wv, int(Nv), lam, bool(coulomb), bool(normalize), params, Sigma, fva.value)


@_preserve_eltype
def ls_windowpsd_lpv(Y, X, V, w, Nv, nw=10, noverlap=0, *, coulomb=False, normalize=True, ctx=None, **kw):
    """ls_windowpsd_lpv(Y,X,V,w,Nv,nw=10,noverlap=0; kwargs...) (src/lsfft.jl:267-277): rect windows (Windows3), one
    ls_spectral_lpv per window on the window's own basis centres, S = Σ_windows |Σ_k x[f,k]|², not normalised.  The
    signals go to the device once; windows are sample ranges (lpvs_ls_windowpsd_lpv)."""
    lam = _lam(kw, 1e-8)
    if kw:
        raise TypeError(f"unexpected keyword arguments {sorted(kw)}")
    ctx = ctx or default_context()
    Yv, Xv, Vv, wv = _f64(Y), _f64(X), _f64(V), _f64(w)
    if not (len(Yv) == len(Xv) == len(Vv)):
        raise ValueError("y, t and v has to be the same length")  # src/windows.jl:96
    n = len(Yv) // int(nw)
    Kw = window_count(len(Yv), n, noverlap) if n > 0 else 0
    S = np.zeros(len(wv))
    fva = np.ones(max(Kw, 1))
    K, info = C.c_int64(0), C.c_int(0)
    ctx.check(ctx.lib.lpvs_ls_windowpsd_lpv(ctx.h, _ptr(Yv), _ptr(Xv), _ptr(Vv), len(Yv), _ptr(wv), len(wv), int(Nv),
                                            int(n), int(noverlap), lam, int(bool(coulomb)), int(bool(normalize)),
                                            _ptr(S), _ptr(fva), C.byref(K), C.byref(info)))
    for v in fva[:K.value]:
        if v < 0.9:  # src/lsfft.jl:256, once per window
            import warnings

            warnings.warn(f"Fraction of variance explained = {v}")
    return S


# ---- sparse estimators ------------------------------------------------------------------------------------------


@dataclass
class NormL1:
    """ProximalOperators.NormL1(λ)."""

    λ: float = 1.0


@dataclass
class NormL0:
    """ProximalOperators.NormL0(λ)."""

    λ: float = 1.0


@dataclass
class IndBallL0:
    """ProximalOperators.IndBallL0(r)."""

    r: int = 1


def _prox_desc(proxg):
    if isinstance(proxg, NormL1):
        return L.PROX_L1, float(proxg.λ)
    if isinstance(proxg, NormL0):
        return L.PROX_L0, float(proxg.λ)
    if isinstance(proxg, IndBallL0):
        return L.PROX_BALL_L0, float(proxg.r)
    raise ValueError("proxg must be NormL1, NormL0 or IndBallL0 (no host-side fallback for other operators)")


def prox(proxg, v, gamma, Nf, zero_first, ctx: Optional[Context] = None):
    """prox!(z, proxg, v, gamma) on the device, with the ADMM loop's own routines (lpvs_prox_fourier): v in the
    reference's order [cos block; sin block], length 2*Nf - zero_first."""
    ctx = ctx or default_context()
    vv = _f64(v)
    kind, param = _prox_desc(proxg)
    z = np.empty_like(vv)
    ctx.check(ctx.lib.lpvs_prox_fourier(ctx.h, kind, param, float(gamma), _ptr(vv), int(Nf), int(bool(zero_first)),
                                        _ptr(z)))
    return z


class ADMM:
    """Device-resident ADMM state (src/lasso.jl:136-171).  ``run`` reproduces the reference's print/callback
    cadence by chunking the device loop every ``printerval`` iterations (SURVEY H6)."""

    def __init__(self, ctx: Context, handle):
        self.ctx = ctx
        self.h = handle
        self.iters = 0
        self.residual = math.inf
        self.converged = False

    @property
    def size(self):
        return int(self.ctx.lib.lpvs_admm_size(self.h))

    def step(self, max_iters, tol):
        it, res, conv = C.c_int64(0), C.c_double(0.0), C.c_int(0)
        self.ctx.check(self.ctx.lib.lpvs_admm_run(self.h, int(max_iters), float(tol), C.byref(it), C.byref(res),
                                                  C.byref(conv)))
        self.iters += it.value
        self.residual = res.value
        self.converged = bool(conv.value)
        return it.value

    def run(self, iters=10000, tol=1e-5, printerval=100, cb=None, verbose=True):
        while self.iters < iters and not self.converged:
            chunk = min(printerval - self.iters % printerval, iters - self.iters)
            self.step(chunk, tol)
            if self.iters % printerval == 0:  # src/lasso.jl:158-163
                if verbose:
                    print("%d ||x-z||₂ %.10f" % (self.iters, self.residual))
                if cb is not None:
                    cb(*self.get())
            if self.converged and verbose:  # :164-168 (a stop on a print iteration prints the line twice)
                print("%d ||x-z||₂ %.10f" % (self.iters, self.residual))
                print("[ Info: ||x-z||₂ ≤ tol")
        return self

    def get(self):
        n = self.size
        x, z = np.empty(n), np.empty(n)
        self.ctx.check(self.ctx.lib.lpvs_admm_get(self.h, _ptr(x), _ptr(z)))
        return x, z

    def result(self, ncomplex):
        out = np.empty(ncomplex, dtype=np.complex128)
        self.ctx.check(self.ctx.lib.lpvs_admm_result(self.h, _ptr(out)))
        return out

    def timing(self):
        ms, by = C.c_double(), C.c_double()
        self.ctx.lib.lpvs_admm_last_timing(self.h, C.byref(ms), C.byref(by))
        return ms.value, by.value

    def free(self):
        if self.h:
            if getattr(self.ctx, "h", None):  # a closed context has already released its handles
                self.ctx.lib.lpvs_admm_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


@_preserve_eltype
def ls_sparse_spectral(y, t, f=None, W=None, *, init=False, proxg=None, iters=10000, tol=1e-5, printerval=100,
                       cb=None, μ=None, mu=None, verbose=False, ctx=None, return_info=False, _m32=False, **kw):
    """ls_sparse_spectral(y,t,f[,W]; init=false, λ=1, proxg=NormL1(λ), iters, tol, printerval, cb, μ)
    -> (x, f)   (src/lasso.jl:85-126).  The weighted method keeps the reference's sign quirk (Q13)."""
    lam = _lam(kw, 1.0)
    if kw:
        raise TypeError(f"unexpected keyword arguments {sorted(kw)}")
    mu = 0.05 if (μ is None and mu is None) else float(μ if μ is not None else mu)
    if not (0 <= mu <= 1):
        raise AssertionError("μ should be ≤ 1")  # src/lasso.jl:143
    ctx = ctx or default_context()
    yv, tv = _f64(y), _f64(t)
    if len(yv) != len(tv):
        raise ValueError("y and t has to be the same length")
    f_in = default_freqs(tv) if f is None else f
    fv = _f64(f_in)
    check_freq(fv)
    Wv = None if W is None else _f64(W)
    kind, param = _prox_desc(proxg if proxg is not None else NormL1(lam))
    h = C.c_void_p()
    if _m32:
        ctx.set_option(L.OPT_ADMM_M32, 1)
    try:
        ctx.check(ctx.lib.lpvs_admm_create_fourier(ctx.h, _ptr(yv), _ptr(tv), len(yv), _ptr(fv), len(fv), _ptr(Wv), kind,
                                                   param, mu, None, int(bool(init)), lam, C.byref(h)))
    finally:
        if _m32:
            ctx.set_option(L.OPT_ADMM_M32, 0)
    solver = ADMM(ctx, h)
    try:
        solver.run(iters=iters, tol=tol, printerval=printerval, cb=cb, verbose=verbose)
        x = solver.result(len(fv))
        info = dict(iters=solver.iters, residual=solver.residual, converged=solver.converged, timing=solver.timing())
        if return_info:
            xr, zr = solver.get()
            info.update(x=xr, z=zr)
    finally:
        solver.free()
    if return_info:
        return x, f_in, info
    return x, f_in


@_preserve_eltype
def ls_sparse_spectral_lpv(y, X, V, w, Nv, *, coulomb=False, normalize=True, iters=10000, tol=1e-5, printerval=100,
                           cb=None, μ=None, mu=None, verbose=False, ctx=None, return_info=False, _m32=False, **kw):
    """ls_sparse_spectral_lpv(y,X,V,w,Nv; λ=1, coulomb=false, normalize=true, ADMM kwargs) -> SpectralExt
    (src/lasso.jl:27-70): group lasso over frequencies."""
    lam = _lam(kw, 1.0)
    if kw:
        raise TypeError(f"unexpected keyword arguments {sorted(kw)}")
    mu = 0.05 if (μ is None and mu is None) else float(μ if μ is not None else mu)
    if not (0 <= mu <= 1):
        raise AssertionError("μ should be ≤ 1")
    ctx = ctx or default_context()
    yv, Xv, Vv, wv = _f64(y), _f64(X), _f64(V), _f64(w)
    h = C.c_void_p()
    if _m32:
        ctx.set_option(L.OPT_ADMM_M32, 1)
    try:
        ctx.check(ctx.lib.lpvs_admm_create_lpv(ctx.h, _ptr(yv), _ptr(Xv), _ptr(Vv), len(yv), _ptr(wv), len(wv), int(Nv),
                                               int(bool(coulomb)), int(bool(normalize)), lam, mu, C.byref(h)))
    finally:
        if _m32:
            ctx.set_option(L.OPT_ADMM_M32, 0)
    solver = ADMM(ctx, h)
    try:
        solver.run(iters=iters, tol=tol, printerval=printerval, cb=cb, verbose=verbose)
        params = solver.result(len(wv) * int(Nv) * (2 if coulomb else 1))  # Nf * Nvv complex parameters
        info = dict(iters=solver.iters, residual=solver.residual, converged=solver.converged, timing=solver.timing())
        if return_info:
            xr, zr = solver.get()
            info.update(x=xr, z=zr)
    finally:
        solver.free()
    se = SpectralExt(yv, Xv, Vv, wv, int(Nv), lam, bool(coulomb), bool(normalize), params, None)
    if return_info:
        return se, info
    return se
