"""Restatement of the sparse multichannel estimators (ls_sparse_windowpsd_multi, ls_sparse_windowcsd_matrix,
ls_sparse_cohere_matrix) on top of oracle/lpvs_oracle.py: every window and channel through
o.ls_sparse_spectral(..., W, mode="gram"), as the pairwise oracle o.ls_windowcsd(..., estimator=...) runs it, and the
C x C sums z_i conj(z_j) in Julia's order.  Test infrastructure only."""
import numpy as np

from oracle import lpvs_oracle as o


def sparse_matrix_sums(Y, t, freqs, nw=10, noverlap=-1, window_func=o.rect, **kw):
    """Raw (Nf, C, C) sums z_i conj(z_j) over all windows (Julia's unfused order per entry), K, freqs and the (K, C)
    iteration counts and final residuals.  kw: lam / proxg / mu / iters / tol of o.ls_sparse_spectral."""
    Y = np.asarray(Y, dtype=np.float64)
    if Y.ndim == 1:
        Y = Y[:, None]
    t = np.asarray(t, dtype=np.float64)
    n = Y.shape[0] // nw
    if freqs is None:
        freqs = o.default_freqs(t, n)
    freqs = np.asarray(freqs, dtype=np.float64)
    kw = dict(kw, printerval=10 ** 9)
    win = o.Windows((t,) + tuple(Y.T), n, noverlap, window_func)
    C = Y.shape[1]
    S = np.zeros((len(freqs), C, C), dtype=np.complex128)
    its, res = [], []
    for parts in win:
        ti = parts[0]
        X, it_k, res_k = [], [], []
        for c in range(C):
            x, _, info = o.ls_sparse_spectral(parts[1 + c], ti, freqs, win.W, mode="gram", return_info=True, **kw)
            X.append(x)
            it_k.append(info["iters"])
            res_k.append(info["residual"])
        X = np.stack(X, axis=1)
        S += o._mul_conj(X[:, :, None], X[:, None, :])
        its.append(it_k)
        res.append(res_k)
    return S, len(win), freqs, np.array(its, dtype=np.int64).reshape(-1, C), np.array(res).reshape(-1, C)


def ls_sparse_windowpsd_multi(Y, t, freqs=None, nw=8, noverlap=-1, window_func=o.rect, **kw):
    S, K, freqs, _, _ = sparse_matrix_sums(Y, t, freqs, nw, noverlap, window_func, **kw)
    return np.einsum("fii->fi", S).real / float(K) ** 2, freqs


def ls_sparse_windowcsd_matrix(Y, t, freqs=None, nw=10, noverlap=-1, window_func=o.rect, **kw):
    S, K, freqs, _, _ = sparse_matrix_sums(Y, t, freqs, nw, noverlap, window_func, **kw)
    return (S.real / K) + 1j * (S.imag / K), freqs


def ls_sparse_cohere_matrix(Y, t, freqs=None, nw=10, noverlap=-1, **kw):
    S, K, freqs, _, _ = sparse_matrix_sums(Y, t, freqs, nw, noverlap, o.hanning, **kw)
    d = np.einsum("fii->fi", S).real
    return o._abs2(S) / (d[:, None, :] * d[:, :, None]), freqs
