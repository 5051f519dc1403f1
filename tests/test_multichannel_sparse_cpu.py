"""Sparse multichannel estimators without a GPU: the oracle's sparse matrix restatement (tests/oracle_matrix_sparse.py)
against its pairwise windowed estimators with estimator = ls_sparse_spectral, and the window-sharded sparse matrix path at world
size 2 on gloo with the oracle standing in for the per-rank GPU compute.  CPU only."""
import os
import socket

import numpy as np
import torch.multiprocessing as mp

from oracle import lpvs_oracle as o

import oracle_matrix_sparse as oms

KW = dict(lam=0.3, mu=0.05, iters=3000, tol=1e-10)


def _record(N, C, seed):
    rng = np.random.default_rng(seed)
    t = np.sort(10 * rng.random(N))
    base = np.sin(2 * np.pi * 1.7 * t)
    Y = np.stack([(0.5 + c) * base + np.cos(2 * np.pi * (0.9 + 0.4 * c) * t) + 0.3 * rng.standard_normal(N)
                  for c in range(C)], axis=1)
    return t, Y


def _est(yi, ti, fr, W, **k):
    return o.ls_sparse_spectral(yi, ti, fr, W, mode="gram", printerval=10 ** 9, **k)


def test_sparse_matrix_oracle_equals_pairwise_oracle():
    """Entry by entry, bit for bit: both run the same per-window ADMM and Julia's unfused accumulation."""
    t, Y = _record(900, 3, 2)
    n, nov = 300, 150
    f = np.arange(1, 12) * 1.0 / (t[n] - t[0])
    for pg in (o.NormL1(0.3), o.NormL0(0.02), o.IndBallL0(5)):
        kw = dict(KW, proxg=pg)
        S, _ = oms.ls_sparse_windowcsd_matrix(Y, t, f, nw=3, noverlap=nov, window_func=o.hanning, **kw)
        Co, _ = oms.ls_sparse_cohere_matrix(Y, t, f, nw=3, noverlap=nov, **kw)
        P, _ = oms.ls_sparse_windowpsd_multi(Y, t, f, nw=3, noverlap=nov, window_func=o.hanning, **kw)
        for i in range(3):
            Pi, _ = o.ls_windowpsd(Y[:, i], t, f, nw=3, noverlap=nov, window_func=o.hanning, estimator=_est, **kw)
            assert np.array_equal(P[:, i], Pi)
            for j in range(3):
                Sij, _ = o.ls_windowcsd(Y[:, i], Y[:, j], t, f, nw=3, noverlap=nov, window_func=o.hanning,
                                        estimator=_est, **kw)
                Cij, _ = o.ls_cohere(Y[:, i], Y[:, j], t, f, nw=3, noverlap=nov, estimator=_est, **kw)
                assert np.array_equal(S[:, i, j], Sij)
                assert np.array_equal(Co[:, i, j], Cij, equal_nan=True)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _oracle_sparse_sums(Y, t, f, W, n, noverlap, proxg, mu, iters, tol, k0, k1, ctx=None):
    hop = n - noverlap
    Yr = Y[k0 * hop:(k1 - 1) * hop + n]
    tr = t[k0 * hop:(k1 - 1) * hop + n]
    S, K, _, _, _ = oms.sparse_matrix_sums(Yr, tr, f, nw=len(Yr) // n, noverlap=noverlap, window_func=lambda m: W,
                                          proxg=proxg, mu=mu, iters=iters, tol=tol)
    assert K == k1 - k0
    return S


def _worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from lpvspectral_jl_b200 import _api as A
    from lpvspectral_jl_b200 import _dist as D

    A.window_matrix_sparse_sums = _oracle_sparse_sums  # the oracle in place of the per-rank GPU call
    t, Y = _record(1500, 3, 8)
    n = 150
    f = np.arange(1, 8) * 2.0 / (t[n] - t[0])
    out = {}
    for kind in (0, 1, 2):
        out[kind] = D.ls_window_matrix_sparse_sharded(kind, Y, t, f, n=n, noverlap=0, W=o.hanning(n),
                                                      proxg=o.NormL1(0.3), mu=0.05, iters=3000, tol=1e-10)
    if rank == 0:
        q.put(out)
    dist.barrier()
    dist.destroy_process_group()


def test_window_matrix_sparse_sharding_world2():
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
    t, Y = _record(1500, 3, 8)
    n = 150
    f = np.arange(1, 8) * 2.0 / (t[n] - t[0])
    kw = dict(proxg=o.NormL1(0.3), mu=0.05, iters=3000, tol=1e-10)
    P, _ = oms.ls_sparse_windowpsd_multi(Y, t, f, nw=10, noverlap=0, window_func=o.hanning, **kw)
    S, _ = oms.ls_sparse_windowcsd_matrix(Y, t, f, nw=10, noverlap=0, window_func=o.hanning, **kw)
    Co, _ = oms.ls_sparse_cohere_matrix(Y, t, f, nw=10, noverlap=0, **kw)
    assert out[0][1] == 10
    for got, ref in ((out[0][0], P), (out[1][0], S), (out[2][0], Co)):
        assert np.linalg.norm(got - ref) <= 1e-13 * np.linalg.norm(ref)
