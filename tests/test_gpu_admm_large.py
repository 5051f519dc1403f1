"""ADMM (ls_sparse_spectral, ls_sparse_spectral_lpv) past the old 25 344-unknown bound: the tiled SYMV plan (-m gpu).

The reference is the oracle's formulas restated in torch FP64 on the GPU (numpy takes minutes at these sizes): the
regressor of oracle.get_fourier_regressor / oracle.lpv_regressor with the reference's phase rounding fl(fl(2 pi f) t) and
column order, M = (G + I/mu)^-1, the ADMM recurrence of src/lasso.jl:136-171 and the prox operators of
oracle/lpvs_oracle.py.  The library's handle and workspaces are released before the torch side is built."""
import math

import numpy as np
import pytest

from oracle import lpvs_oracle as o

pytestmark = pytest.mark.gpu

MU = 0.05
NF = 13120  # with f[0] = 0: Nreg = 26 239, padded to Np = 26 240 (205 blocks of 128), the tiled plan
NP = 26240


def symv_plan(Np, max_item=0):
    """The SYMV plan admm_finish_create picks: the column plan while the whole-vector partial of the old kernel,
    8 (Np + 16*128 + max_item) bytes, fits 220 KB (Np <= 26 112 without groups), else the tiled plan."""
    return "tiled" if 8 * (Np + 16 * 128 + max_item) > 220 * 1024 else "column"


@pytest.fixture(scope="module")
def torch():
    import torch

    return torch


def fourier_problem(Nf=NF, N=8192, zero=True, seed=21, jitter=False):
    """N irregular samples, a few on-grid tones at phase ~pi/4 (cos and sin parts both large) plus 0.01 noise.  jitter:
    t = n + U(0, 0.25), on which the frequency grid is nearly orthogonal (with N = 2 Nf, G is well conditioned)."""
    rng = np.random.default_rng(seed)
    t = (np.arange(N) + 0.25 * rng.random(N)) if jitter else np.sort(N * rng.random(N))
    f = np.arange(0 if zero else 1, Nf + (0 if zero else 1)) / (2.0 * Nf)
    ks = (Nf // 9, Nf // 4, Nf // 3, Nf // 2 + 7, 4 * Nf // 5)
    y = sum((1.0 + 0.2 * i) * np.cos(2 * np.pi * f[k] * t + 0.8 + 0.1 * i) for i, k in enumerate(ks))
    y = y + 0.01 * rng.standard_normal(N)
    return t, y, f, len(ks)


def fourier_regressor(torch, t, f):
    """oracle.get_fourier_regressor on the GPU: [cos | -sin (without the zero frequency)] / sqrt(2 Nf)."""
    tt = torch.as_tensor(t, dtype=torch.float64, device="cuda")
    w = torch.as_tensor((2.0 * np.pi) * np.asarray(f), dtype=torch.float64, device="cuda")  # fl(2 pi f)
    phi = tt[:, None] * w[None, :]
    dd = 1.0 / math.sqrt(2 * len(f))
    C = torch.cos(phi) * dd
    S = -torch.sin(phi) * dd
    if f[0] == 0:
        S = S[:, 1:]
    return torch.cat([C, S], dim=1)


def inverse(torch, G):
    """(G + I/mu)^-1 by Cholesky, G consumed."""
    G.diagonal().add_(1.0 / MU)
    Lc = torch.linalg.cholesky(G)
    del G
    M = torch.cholesky_inverse(Lc)
    del Lc
    return M


def prox(torch, kind, v, param, margins):
    if kind == "l1":
        return torch.sign(v) * torch.clamp(v.abs() - MU * param, min=0.0)
    if kind == "l0":
        thr = math.sqrt(2.0 * MU * param)
        margins.append(float(((v.abs() - thr).abs() / thr).min()))
        return torch.where(v.abs() > thr, v, torch.zeros_like(v))
    if kind == "ball":
        r = int(param)
        a = v.abs()
        srt = torch.sort(a, descending=True).values
        margins.append(float((srt[r - 1] - srt[r]) / srt[r - 1]))
        order = torch.argsort(-a, stable=True)[:r]
        z = torch.zeros_like(v)
        z[order] = v[order]
        return z
    if kind == "group":
        lam, gsize = param
        g = v.view(-1, gsize)
        nrm = torch.sqrt((g * g).sum(dim=1))
        scale = torch.where(nrm > 0, torch.clamp(1.0 - MU * lam / nrm, min=0.0), torch.zeros_like(nrm))
        return (g * scale[:, None]).reshape(-1)
    raise ValueError(kind)


def admm(torch, M, b, quad, kind, param, iters, tol, x0=None):
    """src/lasso.jl:136-171 with the exact x-update x = M rhs; returns (z, x, iterations, last ||x - z||, prox margins)."""
    x = torch.zeros_like(b) if x0 is None else x0.clone()
    z = x.clone()
    u = torch.zeros_like(b)
    margins = []
    nxz, done = math.inf, 0
    for i in range(1, iters + 1):
        v = z - u
        x = torch.mv(M, (v / MU - b) if quad else (b + v / MU))
        z = prox(torch, kind, x + u, param, margins)
        d = x - z
        u = u + d
        nxz = float(torch.sqrt(d @ d))
        done = i
        if nxz < tol:
            break
    return z.cpu().numpy(), x.cpu().numpy(), done, nxz, margins


def reference_fourier(torch, t, y, f, W=None, x0=None):
    """b and M of the Fourier problem: LeastSquares (b = A'y) or, with W, Quadratic (b = A'Wy, Q13 sign in admm())."""
    A = fourier_regressor(torch, t, f)
    yy = torch.as_tensor(y, dtype=torch.float64, device="cuda")
    if W is None:
        b = A.T @ yy
        G = A.T @ A
    else:
        AtW = A.T * torch.as_tensor(W, dtype=torch.float64, device="cuda")[None, :]
        b = AtW @ yy
        G = AtW @ A
        del AtW
    ridge = None
    if x0 == "ridge":  # fourier_solve(A, y, zerofreq, lambda = 1): (A'A + I) x = A'y, the unweighted start (Q14)
        Gr = (A.T @ A)
        Gr.diagonal().add_(1.0)
        ridge = torch.linalg.solve(Gr, A.T @ yy)
        del Gr
    del A
    return inverse(torch, G), b, ridge


def free_all(ctx, torch):
    ctx.release_workspace()
    torch.cuda.empty_cache()


def max_err(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))))


def support(z):
    return set(np.flatnonzero(z).tolist())


_REF = {}


def ref_M(torch, key, build):
    if key not in _REF:
        _REF.clear()
        torch.cuda.empty_cache()
        _REF[key] = build()
    return _REF[key]


# every prox, unweighted and weighted, on the tiled plan; plus Np = 25 600, above the old bound on the column plan
@pytest.mark.parametrize("Nf,kind,weighted", [(NF, k, w) for k in ("l1", "l0", "ball") for w in (False, True)]
                         + [(12800, "l1", False)])
def test_fourier_fixed_iterations(ctx, torch, Nf, kind, weighted):
    import lpvspectral_jl_b200 as lp

    assert symv_plan(2 * Nf) == ("tiled" if Nf == NF else "column")
    t, y, f, ntones = fourier_problem(Nf=Nf)
    W = (o.hanning(len(t)) + 0.1) if weighted else None
    param = {"l1": 1.0, "l0": 0.5, "ball": 2 * ntones}[kind]
    pg = {"l1": lp.NormL1, "l0": lp.NormL0, "ball": lp.IndBallL0}[kind](param)
    _, _, info = lp.ls_sparse_spectral(y, t, f, W, proxg=pg, iters=150, tol=0.0, printerval=150, ctx=ctx,
                                       return_info=True)
    assert info["iters"] == 150
    free_all(ctx, torch)
    M, b, _ = ref_M(torch, ("fourier", Nf, weighted), lambda: reference_fourier(torch, t, y, f, W))
    z, _, its, _, margins = admm(torch, M, b, weighted, kind, param, 150, 0.0)
    assert its == 150
    assert max_err(info["z"], z) <= 1e-9 * np.max(np.abs(z))
    if kind != "l1":
        # no |x + u| within 1e-6 relative of the threshold / the r-th largest value in any iteration: no tie can flip
        assert min(margins) > 1e-6
        assert support(info["z"]) == support(z)
        assert len(support(z)) > 0


def test_fourier_stop_test_chunks_repeat_and_init(ctx, torch):
    import lpvspectral_jl_b200 as lp

    # well conditioned (N = Np jittered samples), so that the stop test is reached in a few hundred iterations; on the
    # underdetermined problems above the null space of G contracts by only 1/(1 + mu lambda_min) per iteration
    t, y, f, _ = fourier_problem(N=NP, seed=24, jitter=True)
    assert symv_plan(NP) == "tiled"
    tol, cap = 1e-5, 20000
    kw = dict(proxg=lp.NormL1(1.0), iters=cap, tol=tol, ctx=ctx, return_info=True)
    _, _, one = lp.ls_sparse_spectral(y, t, f, printerval=cap, **kw)
    _, _, chunked = lp.ls_sparse_spectral(y, t, f, printerval=37, **kw)
    _, _, again = lp.ls_sparse_spectral(y, t, f, printerval=cap, **kw)
    assert one["converged"] and one["residual"] < tol
    for other in (chunked, again):
        assert other["iters"] == one["iters"] and other["residual"] == one["residual"]
        assert np.array_equal(other["z"], one["z"]) and np.array_equal(other["x"], one["x"])
    _, _, ini = lp.ls_sparse_spectral(y, t, f, init=True, proxg=lp.NormL1(1.0), iters=150, tol=0.0, printerval=150,
                                      ctx=ctx, return_info=True)
    free_all(ctx, torch)
    M, b, ridge = ref_M(torch, ("fourier-ridge",), lambda: reference_fourier(torch, t, y, f, None, "ridge"))
    z, _, its, nxz, _ = admm(torch, M, b, False, "l1", 1.0, cap, tol)
    assert abs(its - one["iters"]) <= 1
    assert nxz < tol
    assert max_err(one["z"], z) <= 1e-9 * np.max(np.abs(z))
    z0, _, _, _, _ = admm(torch, M, b, False, "l1", 1.0, 150, 0.0, x0=ridge)
    assert max_err(ini["z"], z0) <= 1e-9 * np.max(np.abs(z0))


def test_lpv_group_lasso_above_old_bound(ctx, torch):
    import lpvspectral_jl_b200 as lp

    Nf, Nv, N, lam = 1640, 8, 4096, 5.0
    assert symv_plan(2 * Nf * Nv, 2 * Nv) == "tiled"
    Y, V, X = o.generate_lpv_signal(N, seed=4)
    w = 2 * np.pi * np.arange(1, Nf + 1) * 0.05  # 0.05 .. 82 Hz: holds the 2, 10 and 20 Hz components
    se, info = lp.ls_sparse_spectral_lpv(Y, X, V, w, Nv, lam=lam, coulomb=False, iters=150, tol=0.0, printerval=150,
                                         ctx=ctx, return_info=True)
    assert len(info["z"]) == 2 * Nf * Nv == NP
    free_all(ctx, torch)
    _REF.clear()
    K = torch.as_tensor(o.basis_activation(V, Nv, True, False), dtype=torch.float64, device="cuda")  # N x Nv
    ph = torch.as_tensor(X, dtype=torch.float64, device="cuda")[:, None] * torch.as_tensor(w, dtype=torch.float64,
                                                                                           device="cuda")[None, :]
    re = (K[:, :, None] * torch.cos(ph)[:, None, :]).reshape(N, -1)  # column f + k Nf (oracle.lpv_regressor)
    im = (K[:, :, None] * (-torch.sin(ph))[:, None, :]).reshape(N, -1)
    Ar = torch.cat([re, im], dim=1)
    del re, im, ph
    Phi = Ar[:, torch.as_tensor(o.lpv_group_perm(Nf, Ar.shape[1]), device="cuda")]
    del Ar
    yy = torch.as_tensor(Y, dtype=torch.float64, device="cuda")
    b = Phi.T @ yy
    M = inverse(torch, Phi.T @ Phi)
    del Phi
    z, _, _, _, _ = admm(torch, M, b, False, "group", (lam, 2 * Nv), 150, 0.0)
    del M
    torch.cuda.empty_cache()
    assert max_err(info["z"], z) <= 1e-9 * np.max(np.abs(z))
    assert support(info["z"]) == support(z)


def test_m32_matches_fp64(ctx):
    import lpvspectral_jl_b200 as lp

    assert symv_plan(NP) == "tiled"
    t, y, f, ntones = fourier_problem(seed=22)
    y32 = y.astype(np.float32)
    pg = lp.IndBallL0(2 * ntones)
    _, _, i64 = lp.ls_sparse_spectral(y32.astype(np.float64), t, f, proxg=pg, iters=150, tol=0.0, printerval=150,
                                      ctx=ctx, return_info=True)
    _, _, i32 = lp.ls_sparse_spectral(y32, t, f, proxg=pg, iters=150, tol=0.0, printerval=150, ctx=ctx,
                                      return_info=True)
    ctx.release_workspace()
    assert support(i32["z"]) == support(i64["z"])
    assert max_err(i32["z"], i64["z"]) <= 1e-5 * np.max(np.abs(i64["z"]))


def test_fourier_past_int32_elements(ctx, torch):
    """Np = 46 464: Np^2 > 2^31 elements of G, of the inverse and of its single-precision copy."""
    import lpvspectral_jl_b200 as lp

    t, y, f, _ = fourier_problem(Nf=23232, zero=False, seed=23)
    y = y.astype(np.float32).astype(np.float64)  # the same input for the FP64 run and the Float32 (M32) run
    kw = dict(proxg=lp.NormL1(1.0), iters=50, tol=0.0, printerval=50, ctx=ctx, return_info=True)
    _, _, info = lp.ls_sparse_spectral(y, t, f, **kw)
    _, _, i32 = lp.ls_sparse_spectral(y.astype(np.float32), t, f, **kw)
    assert len(info["z"]) == 46464
    assert max_err(i32["z"], info["z"]) <= 1e-5 * np.max(np.abs(info["z"]))
    free_all(ctx, torch)
    _REF.clear()
    M, b, _ = reference_fourier(torch, t, y, f)
    z, _, _, _, _ = admm(torch, M, b, False, "l1", 1.0, 50, 0.0)
    del M, b
    torch.cuda.empty_cache()
    assert max_err(info["z"], z) <= 1e-9 * np.max(np.abs(z))


def test_errors_gemv_and_memory(ctx, torch):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    t, y, f, _ = fourier_problem()
    ctx.set_option(L.OPT_ADMM_SYMV, 0)
    try:
        with pytest.raises(NotImplementedError, match="GEMV"):
            lp.ls_sparse_spectral(y, t, f, iters=10, ctx=ctx)
    finally:
        ctx.set_option(L.OPT_ADMM_SYMV, -1)
    # G and its inverse (16 Np^2 = 11 GB) cannot fit next to a filler that leaves 4 GB free
    _REF.clear()
    free_all(ctx, torch)
    free_b, _ = torch.cuda.mem_get_info()
    filler = torch.empty(max(0, free_b - (4 << 30)), dtype=torch.uint8, device="cuda")
    try:
        with pytest.raises(MemoryError, match="Np=%d" % NP):
            lp.ls_sparse_spectral(y, t, f, iters=10, ctx=ctx)
    finally:
        del filler
        torch.cuda.empty_cache()
    # the context still solves a small problem correctly
    rng = np.random.default_rng(7)
    ts = np.sort(10.0 * rng.random(800))
    ys = np.sin(2 * np.pi * 3.0 * ts) + 0.7 * np.cos(2 * np.pi * 7.5 * ts + 0.3) + 0.1 * rng.standard_normal(800)
    fs = np.arange(0, 161) * 0.1
    kw = dict(iters=3000, tol=1e-9, mu=MU)
    x, _, info = lp.ls_sparse_spectral(ys, ts, fs, proxg=lp.NormL1(0.5), ctx=ctx, return_info=True, **kw)
    xr, _, ri = o.ls_sparse_spectral(ys, ts, fs, proxg=o.NormL1(0.5), mode="gram", return_info=True,
                                     printerval=10 ** 9, **kw)
    assert info["iters"] == ri["iters"]
    assert np.linalg.norm(x - xr) <= 1e-9 * np.linalg.norm(xr)
