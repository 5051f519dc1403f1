"""Literal-mode restatement of the multichannel estimators (ls_windowpsd_multi, ls_windowcsd_matrix, ls_cohere_matrix) on top
of oracle/lpvs_oracle.py: per window ONE LU factorisation of A'WA + lam I with the N right-hand sides A'W (the reference's
`(A'Wd*A + lam I) \\ (A'Wd)`, src/lsfft.jl:77), applied to every channel.  Test infrastructure only."""
import numpy as np
import scipy.linalg as sla

from oracle import lpvs_oracle as o


def _window_coeffs(Y, t, freqs, nw, noverlap, window_func, lam, jitter=False):
    """Yields the (Nf, C) complex coefficients of every window.  jitter: a window whose A'WA + lam I is not positive definite
    (numpy's Cholesky fails) is solved with the ridge max(lam, Nreg eps max diag A'WA) instead, the library's retry."""
    Y = np.asarray(Y, dtype=np.float64)
    if Y.ndim == 1:
        Y = Y[:, None]
    t = np.asarray(t, dtype=np.float64)
    n = Y.shape[0] // nw
    if freqs is None:
        freqs = o.default_freqs(t, n)
    freqs = np.asarray(freqs, dtype=np.float64)
    win = o.Windows((t,) + tuple(Y.T), n, noverlap, window_func)

    def gen():
        for parts in win:
            ti, Yi = parts[0], np.stack(parts[1:], axis=1)
            A, zerofreq = o.get_fourier_regressor(ti, freqs)
            AtW = A.T * win.W[None, :]
            G = AtW @ A
            M = G + lam * np.eye(A.shape[1])
            if jitter:
                try:
                    np.linalg.cholesky(M)
                except np.linalg.LinAlgError:
                    M = G + max(lam, A.shape[1] * np.finfo(np.float64).eps * np.diag(G).max()) * np.eye(A.shape[1])
            lu = sla.lu_factor(M, check_finite=False)
            P = sla.lu_solve(lu, AtW, check_finite=False)
            Xr = P @ Yi
            yield np.stack([o.fourier2complex(Xr[:, c], zerofreq) for c in range(Yi.shape[1])], axis=1)

    return gen(), len(win), freqs, Y.shape[1]


def matrix_sums(Y, t, freqs, nw=10, noverlap=-1, window_func=o.rect, lam=1e-10, jitter=False):
    """Raw (Nf, C, C) sums x_i conj(x_j) over all windows, Julia's unfused order per entry."""
    gen, K, freqs, C = _window_coeffs(Y, t, freqs, nw, noverlap, window_func, lam, jitter)
    S = np.zeros((len(freqs), C, C), dtype=np.complex128)
    for X in gen:
        S += o._mul_conj(X[:, :, None], X[:, None, :])  # entry (i, j): x_i conj(x_j), elementwise as the pairwise loop
    return S, K, freqs


def ls_windowpsd_multi(Y, t, freqs=None, nw=8, noverlap=-1, window_func=o.rect, lam=1e-10):
    gen, K, freqs, C = _window_coeffs(Y, t, freqs, nw, noverlap, window_func, lam)
    S = np.zeros((len(freqs), C))
    for X in gen:
        S += o._abs2(X)
    return S / float(K) ** 2, freqs


def ls_windowcsd_matrix(Y, t, freqs=None, nw=10, noverlap=-1, window_func=o.rect, lam=1e-10):
    S, K, freqs = matrix_sums(Y, t, freqs, nw, noverlap, window_func, lam)
    return (S.real / K) + 1j * (S.imag / K), freqs


def ls_cohere_matrix(Y, t, freqs=None, nw=10, noverlap=-1, lam=1e-10):
    S, K, freqs = matrix_sums(Y, t, freqs, nw, noverlap, o.hanning, lam)
    d = np.einsum("fii->fi", S).real
    return o._abs2(S) / (d[:, None, :] * d[:, :, None]), freqs
