"""Multichannel estimators without a GPU: the literal oracle's matrix estimators against its pairwise ones,
lpvs_ls_window_matrix_finalize on hand-built sums, and the window-sharded matrix path at world size 2 on gloo with the
oracle standing in for the per-rank GPU compute.  CPU only."""
import os
import socket

import numpy as np
import pytest
import torch.multiprocessing as mp

from oracle import lpvs_oracle as o

import oracle_matrix as om


def _record(N=1800, C=3, seed=4):
    rng = np.random.default_rng(seed)
    t = np.sort(10 * rng.random(N))
    base = np.sin(2 * np.pi * 7 * t)
    Y = np.stack([(0.5 + c) * base + np.cos(2 * np.pi * (3 + c) * t) + 0.3 * rng.standard_normal(N) for c in range(C)],
                 axis=1)
    return t, Y


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(b).max()


def test_oracle_matrix_equals_pairwise_oracle():
    t, Y = _record()
    nw = 6
    n = len(t) // nw
    f = np.arange(10) * 2.0 / (t[n] - t[0])
    S, _ = om.ls_windowcsd_matrix(Y, t, f, nw=nw, window_func=o.hanning)
    Co, _ = om.ls_cohere_matrix(Y, t, f, nw=nw)
    P, _ = om.ls_windowpsd_multi(Y, t, f, nw=nw, window_func=o.hanning)
    for i in range(Y.shape[1]):
        Pr, _ = o.ls_windowpsd(Y[:, i], t, f, nw=nw, window_func=o.hanning)
        assert _rel(P[:, i], Pr) <= 1e-13
        for j in range(Y.shape[1]):
            Sr, _ = o.ls_windowcsd(Y[:, i], Y[:, j], t, f, nw=nw, window_func=o.hanning)
            Cr, _ = o.ls_cohere(Y[:, i], Y[:, j], t, f, nw=nw)
            assert _rel(S[:, i, j], Sr) <= 1e-13
            assert _rel(Co[:, i, j], Cr) <= 1e-13


def _channel_inputs():
    rng = np.random.default_rng(3)
    F = np.asfortranarray(rng.standard_normal((2500, 5)))  # N not a multiple of the 1024-row transpose blocks
    return {
        "fortran": F,
        "c_order": np.ascontiguousarray(F),
        "c_order_small_n": np.ascontiguousarray(F[:700]),  # N < 1024: one partial block
        "c_order_n2048": np.ascontiguousarray(rng.standard_normal((2048, 3))),  # whole blocks only
        "rows_strided": F[::2],
        "columns_strided": np.ascontiguousarray(F)[:, ::2],
        "fortran_columns_strided": F[:, ::2],
        "float32": np.ascontiguousarray(F).astype(np.float32),
        "float32_fortran": F.astype(np.float32, order="F"),
        "one_column_c_order": np.ascontiguousarray(F[:, 2:3]),
        "one_d": F[:, 1].copy(),
    }


@pytest.mark.parametrize("name", list(_channel_inputs()))
def test_channels_layout(name):
    """_api._channels: C x N contiguous float64, channel c = Y[:, c], whatever the order, strides and dtype of Y."""
    from lpvspectral_jl_b200 import _api

    Y = _channel_inputs()[name]
    out = _api._channels(Y)
    want = np.ascontiguousarray(np.asarray(Y, dtype=np.float64).reshape(len(Y), -1).T)
    assert out.dtype == np.float64 and out.flags.c_contiguous
    assert np.array_equal(out, want) and out.shape == want.shape


def test_matrix_finalize_normalisations():
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    rng = np.random.default_rng(1)
    Nf, C, K = 5, 3, 7
    Z = rng.standard_normal((Nf, C, C)) + 1j * rng.standard_normal((Nf, C, C))
    S = Z @ np.conj(np.transpose(Z, (0, 2, 1)))  # Hermitian, positive diagonal
    d = np.einsum("fii->fi", S).real
    psd = lp.window_matrix_finalize(L.WIN_PSD, S, K)
    csd = lp.window_matrix_finalize(L.WIN_CSD, S, K)
    coh = lp.window_matrix_finalize(L.WIN_COHERE, S, K)
    assert psd.shape == (Nf, C) and np.array_equal(psd, d / float(K) ** 2)
    assert csd.dtype == np.complex128 and np.array_equal(csd, S.real / K + 1j * (S.imag / K))
    want = (S.real * S.real + S.imag * S.imag) / (d[:, None, :] * d[:, :, None])
    assert np.array_equal(coh, want)
    assert np.all(np.einsum("fii->fi", coh) == 1.0)
    for kind in (L.WIN_PSD, L.WIN_CSD, L.WIN_COHERE):  # K = 0: 0/0, as lpvs_ls_window_finalize
        assert np.all(np.isnan(lp.window_matrix_finalize(kind, np.zeros((Nf, C, C), dtype=np.complex128), 0)))
    with pytest.raises(ValueError):
        lp.window_matrix_finalize(7, S, K)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _oracle_matrix_sums(Y, t, f, W, n, noverlap, lam, k0, k1):
    hop = n - noverlap
    Yr = Y[k0 * hop:(k1 - 1) * hop + n]
    tr = t[k0 * hop:(k1 - 1) * hop + n]
    # the oracle cuts windows of len(Yr) // nw samples: nw chosen so that is exactly n
    S, K, _ = om.matrix_sums(Yr, tr, f, nw=len(Yr) // n, noverlap=noverlap, window_func=lambda m: W, lam=lam)
    assert K == k1 - k0
    return S


def _worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from lpvspectral_jl_b200 import _dist as D

    t, Y = _record(N=2000, C=3, seed=8)
    n = 200
    f = np.arange(9) * 2.0 / (t[n] - t[0])
    out = {}
    for kind in (0, 1, 2):
        W = o.hanning(n)
        out[kind] = D.ls_window_matrix_sharded(kind, Y, t, f, n=n, noverlap=0, W=W, lam=1e-10,
                                               sums_fn=_oracle_matrix_sums)
    if rank == 0:
        q.put(out)
    dist.barrier()
    dist.destroy_process_group()


def test_window_matrix_sharding_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    t, Y = _record(N=2000, C=3, seed=8)
    n = 200
    f = np.arange(9) * 2.0 / (t[n] - t[0])
    P, _ = om.ls_windowpsd_multi(Y, t, f, nw=10, noverlap=0, window_func=o.hanning)
    S, _ = om.ls_windowcsd_matrix(Y, t, f, nw=10, noverlap=0, window_func=o.hanning)
    Co, _ = om.ls_cohere_matrix(Y, t, f, nw=10, noverlap=0)
    assert out[0][1] == 10
    assert _rel(out[0][0], P) <= 1e-13
    assert _rel(out[1][0], S) <= 1e-13
    assert _rel(out[2][0], Co) <= 1e-13
