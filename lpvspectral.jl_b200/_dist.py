"""Multi-GPU host logic (one process per GPU, torch.distributed for the plumbing only).

Two sharding modes, as the path allows (SURVEY 8e):

* windows are independent units -> contiguous window ranges per rank, NO data-path collective; only the
  Nf-long accumulators are summed once at the end (``ls_window_sharded``);
* one very tall problem -> contiguous row blocks per rank, each forms its partial Gram on device, ONE
  all-reduce (NCCL over NVLink) of the packed Gram + right-hand sides, then the factorisation
  (``ls_spectral_rowsharded``).

The compute callables are injectable so the sharding / reduction logic can be exercised with the ``gloo`` backend
on CPU (tests/test_dist_gloo.py); the defaults call liblpvs on the rank's GPU.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Optional

import numpy as np

from . import _api as A
from . import _lib as L

__all__ = ["shard_range", "ls_window_sharded", "ls_window_matrix_sharded", "ls_window_sparse_sharded",
           "ls_spectral_rowsharded", "admm_shard"]


def shard_range(K: int, rank: int, world: int):
    """Contiguous range [K*r/P, K*(r+1)/P) of units for rank r."""
    return (K * rank) // world, (K * (rank + 1)) // world


def _world(group=None):
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def _allreduce_sum_np(arr: np.ndarray, group=None, device=None) -> np.ndarray:
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return arr
    tt = torch.from_numpy(np.ascontiguousarray(arr))
    if device is not None:
        tt = tt.to(device)
    dist.all_reduce(tt, op=dist.ReduceOp.SUM, group=group)
    return tt.cpu().numpy()


def _raise_together(err: Optional[BaseException], group=None, device=None):
    """A rank-local failure (NOT_SPD in one window range, NONFINITE, NOMEM) must not leave the other ranks blocked in the
    data all-reduce until the NCCL timeout: every rank first all-reduces a status flag and all of them raise."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        if err is not None:
            raise err
        return
    flag = torch.tensor([1.0 if err is not None else 0.0], dtype=torch.float64)
    if device is not None:
        flag = flag.to(device)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
    if err is not None:
        raise err
    if float(flag.item()) > 0:
        raise RuntimeError("a sharded liblpvs call failed on another rank (see that rank's exception)")


def ls_window_sharded(kind, y, u, t, freqs, *, n, noverlap=-1, W, lam=1e-10, ctx: Optional[A.Context] = None,
                      group=None, sums_fn: Optional[Callable] = None, reduce_device=None):
    """Windowed PSD/CSD/coherence with the windows sharded across ranks.

    Every rank passes the same full arrays; only its window range's samples travel to its GPU.  Returns the
    finalised estimate on every rank.  ``sums_fn(kind, y, u, t, freqs, W, n, noverlap, lam, k0, k1)`` defaults to
    the liblpvs call."""
    rank, world = _world(group)
    if noverlap < 0:
        noverlap = n >> 1
    K = A.window_count(len(y), n, noverlap)
    k0, k1 = shard_range(K, rank, world)
    if sums_fn is None:
        sums_fn = lambda *a: A.window_sums(*a, ctx=ctx)  # noqa: E731
    nf = len(freqs)
    slen = {L.WIN_PSD: 1, L.WIN_CSD: 2, L.WIN_COHERE: 4}[kind] * nf
    err = None
    try:
        sums = sums_fn(kind, y, u, t, freqs, W, n, noverlap, lam, k0, k1) if k1 > k0 else np.zeros(slen)
    except Exception as e:  # noqa: BLE001 -- re-raised on every rank below
        err, sums = e, np.zeros(slen)
    _raise_together(err, group, reduce_device)
    sums = _allreduce_sum_np(np.asarray(sums, dtype=np.float64), group, reduce_device)
    return A.window_finalize(kind, sums, nf, K), K


def ls_window_matrix_sharded(kind, Y, t, freqs, *, n, noverlap=-1, W, lam=1e-10, ctx: Optional[A.Context] = None,
                             group=None, sums_fn: Optional[Callable] = None, reduce_device=None):
    """ls_windowpsd_multi / ls_windowcsd_matrix / ls_cohere_matrix (by ``kind``) of the N x C matrix Y with the windows
    sharded across ranks: one all-reduce of the Nf x C x C sums at the end.  Returns (estimate, K) on every rank.
    ``sums_fn(Y, t, freqs, W, n, noverlap, lam, k0, k1) -> (Nf, C, C) complex`` defaults to the liblpvs call."""
    rank, world = _world(group)
    if noverlap < 0:
        noverlap = n >> 1
    Yv = np.asarray(Y, dtype=np.float64)
    nch = 1 if Yv.ndim == 1 else Yv.shape[1]
    K = A.window_count(Yv.shape[0], n, noverlap)
    k0, k1 = shard_range(K, rank, world)
    if sums_fn is None:
        sums_fn = lambda *a: A.window_matrix_sums(*a, ctx=ctx)  # noqa: E731
    shape = (len(freqs), nch, nch)
    err = None
    try:
        sums = sums_fn(Yv, t, freqs, W, n, noverlap, lam, k0, k1) if k1 > k0 else np.zeros(shape, dtype=np.complex128)
    except Exception as e:  # noqa: BLE001 -- re-raised on every rank below
        err, sums = e, np.zeros(shape, dtype=np.complex128)
    _raise_together(err, group, reduce_device)
    flat = np.ascontiguousarray(np.asarray(sums, dtype=np.complex128)).view(np.float64)  # interleaved (re, im)
    sums = _allreduce_sum_np(flat, group, reduce_device).view(np.complex128).reshape(shape)
    return A.window_matrix_finalize(kind, sums, K), K


def ls_window_sparse_sharded(kind, y, u, t, freqs, *, n, noverlap=-1, W, proxg, mu=0.05, iters=10000, tol=1e-5,
                             ctx: Optional[A.Context] = None, group=None, reduce_device=None):
    """Windowed estimators with estimator = ls_sparse_spectral, windows sharded across ranks: every window is an
    independent ADMM problem, so as for the dense estimators there is no data-path collective -- one all-reduce of
    the Nf-long accumulators at the end."""
    fn = lambda k, yy, uu, tt, ff, WW, nn, nov, _lam, k0, k1: A.window_sparse_sums(  # noqa: E731
        k, yy, uu, tt, ff, WW, nn, nov, proxg, mu, iters, tol, k0, k1, ctx=ctx)
    return ls_window_sharded(kind, y, u, t, freqs, n=n, noverlap=noverlap, W=W, ctx=ctx, group=group, sums_fn=fn,
                             reduce_device=reduce_device)


def ls_window_matrix_sparse_sharded(kind, Y, t, freqs, *, n, noverlap=-1, W, proxg, mu=0.05, iters=10000, tol=1e-5,
                                    ctx: Optional[A.Context] = None, group=None, reduce_device=None):
    """ls_sparse_windowpsd_multi / ls_sparse_windowcsd_matrix / ls_sparse_cohere_matrix (by ``kind``) with the windows
    sharded across ranks: every (window, channel) is an independent ADMM problem, so there is no data-path collective --
    one all-reduce of the Nf x C x C sums at the end.  Returns (estimate, K) on every rank."""
    fn = lambda YY, tt, ff, WW, nn, nov, _lam, k0, k1: A.window_matrix_sparse_sums(  # noqa: E731
        YY, tt, ff, WW, nn, nov, proxg, mu, iters, tol, k0, k1, ctx=ctx)
    return ls_window_matrix_sharded(kind, Y, t, freqs, n=n, noverlap=noverlap, W=W, ctx=ctx, group=group, sums_fn=fn,
                                    reduce_device=reduce_device)


def ls_spectral_rowsharded(y, t, f, W=None, *, u=None, lam=1e-10, ctx: Optional[A.Context] = None, group=None):
    """Weighted/unweighted ls_spectral for one very tall problem, rows sharded across ranks.

    Each rank forms A_r' W_r A_r and A_r' W_r [y u] on its GPU for its contiguous row block, the packed buffers
    are summed with one NCCL all-reduce, and every rank factorises.  Returns x (Nf complex, or (2, Nf) with u)."""
    import torch
    import torch.distributed as dist

    ctx = ctx or A.default_context()
    rank, world = _world(group)
    yv, tv, fv = A._f64(y), A._f64(t), A._f64(f)
    uv = None if u is None else A._f64(u)
    Wv = None if W is None else A._f64(W)
    N = len(yv)
    r0, r1 = shard_range(N, rank, world)
    dev = torch.device("cuda", ctx.device)
    d_t = torch.from_numpy(tv[r0:r1]).to(dev)
    d_y = torch.from_numpy(yv[r0:r1]).to(dev)
    d_u = None if uv is None else torch.from_numpy(uv[r0:r1]).to(dev)
    d_W = None if Wv is None else torch.from_numpy(Wv[r0:r1]).to(dev)
    npk = int(ctx.lib.lpvs_packed_size(len(fv)))
    packed = torch.empty(npk, dtype=torch.float64, device=dev)
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
    torch.cuda.synchronize(dev)
    err = None
    try:
        ctx.check(ctx.lib.lpvs_gram_partial_dev(ctx.h, p(d_y), p(d_u), p(d_t), p(d_W), r1 - r0, A._ptr(fv), len(fv),
                                                p(packed)))
    except Exception as e:  # noqa: BLE001 -- re-raised on every rank below
        err = e
    _raise_together(err, group, dev)
    if world > 1:
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
        torch.cuda.synchronize(dev)
    nrhs = 1 if uv is None else 2
    ridge = lam if Wv is not None else lam * lam  # Q4 / Q5
    x = np.empty((nrhs, len(fv)), dtype=np.complex128)
    info = C.c_int(0)
    ctx.check(ctx.lib.lpvs_solve_packed_dev(ctx.h, p(packed), A._ptr(fv), len(fv), nrhs, ridge, A._ptr(x),
                                            C.byref(info)))
    return x[0] if nrhs == 1 else x


def admm_shard(solver: "A.ADMM", group=None):
    """Shard ONE ADMM problem over the ranks of a node (every rank must have created the same problem; NormL1 / NormL0, and -- with the default one-exchange scheme -- IndBallL0 and the group prox).

    The loop then runs as a persistent kernel per GPU that exchanges partial products and the new right-hand side with
    device-initiated peer stores over NVLink (lpvs_admm_shard_*); torch.distributed only carries the 64-byte CUDA IPC
    handles and the barriers around the runs.  Call ``dist.barrier()`` after ``solver.step/run`` before reading results."""
    import torch.distributed as dist

    rank, world = _world(group)
    if world < 2:
        return solver
    ctx = solver.ctx
    ctx.check(ctx.lib.lpvs_admm_shard_begin(solver.h, rank, world))
    buf = C.create_string_buffer(64)
    ctx.check(ctx.lib.lpvs_admm_shard_handle(solver.h, C.cast(buf, C.c_void_p)))
    handles = [None] * world
    dist.all_gather_object(handles, bytes(buf.raw), group=group)
    blob = C.create_string_buffer(b"".join(handles), 64 * world)
    ctx.check(ctx.lib.lpvs_admm_shard_connect(solver.h, C.cast(blob, C.c_void_p)))
    dist.barrier(group=group)
    return solver
