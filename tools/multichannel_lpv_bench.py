"""ls_spectral_lpv of C output channels sharing X and V (lpvs_ls_spectral_lpv_multi) against C single-channel
lpvs_ls_spectral_lpv calls.

Shapes: cfg4 (N = 20000, Nf = 64, Nv = 50: 6400 real unknowns) at the reference's default lambda = 1e-8, where the dense
estimator takes the shifted-CholeskyQR route, and a refinement-route shape (N = 4000, Nf = 20, Nv = 20, lambda = 0.02).
Channel c is the shape's LPV output with its own seeded noise.  Both forms return what a user of the estimator gets: the
parameters, Sigma (the multi-channel call returns Sigma0 and var(e_c), from which Sigma_c = var(e_c) Sigma0) and fva.  For C in
{1, 8, 32} each form is warmed up once and timed over --reps calls; the call returns only after its results are on the host.
Every column is compared with its single-channel call.  The stage split of one C = 8 call per shape comes from a
torch.profiler run of its own, kernels grouped by name.  Device name and power limit are read in the same run.

    python tools/multichannel_lpv_bench.py --out profiles/multichannel_lpv_bench.json

--dump DIR saves ls_spectral_multi, ls_spectral_lpv and ls_windowpsd_lpv outputs on seeded inputs, so two builds can be
compared bit for bit; --root imports the package (and its library) from another checkout.

    python tools/multichannel_lpv_bench.py --dump out/branch
    python tools/multichannel_lpv_bench.py --dump out/parent --root /path/to/parent/checkout
"""
import argparse
import ctypes as C
import json
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if "--root" in sys.argv:
    ROOT = os.path.abspath(sys.argv[sys.argv.index("--root") + 1])
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from multichannel_bench import device_info  # noqa: E402

STAGES = [("tables", ("k_lpv_tables",)), ("gram", ("k_gram<", "k_gram(", "k_reduce_parts")), ("rhs", ("k_gram_rhs",)),
          ("factor", ("potf2", "k_gemm_tiles", "k_diag", "k_max_diag", "k_min_pivot", "k_set_shift", "k_pivot")),
          ("trtri", ("k_trtri_rd", "k_copy_diag_inv")), ("qr_objects", ("k_gemm_nt", "k_materialize", "k_transpose_linv")),
          ("sigma", ("potri", "k_potri", "k_gather_ref", "k_trtri", "k_lauum")), ("skinny", ("k_skinny",)),
          ("op_apply", ("k_op_apply",)), ("variance", ("k_sum_sq", "k_sum_parts"))]

SHAPES = {"cfg4_qr": dict(N=20000, Nf=64, Nv=50, lam=1e-8, seed=4, wscale=0.4),
          "refine": dict(N=4000, Nf=20, Nv=20, lam=0.02, seed=5, wscale=1.0)}


def vp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def shape_inputs(sh, nch):
    from oracle import lpvs_oracle as o

    Y0, V, X = o.generate_lpv_signal(sh["N"], seed=sh["seed"])
    w = 2 * np.pi * np.arange(1, sh["Nf"] + 1) * sh["wscale"]
    rng = np.random.default_rng(7)
    Y = np.stack([Y0 + 0.1 * rng.standard_normal(sh["N"]) for _ in range(nch)], axis=1)
    return Y, X, V, w


def dump(outdir):
    """ls_spectral_multi (unweighted and weighted), ls_spectral_lpv (with Sigma, two lambdas, coulomb) and
    ls_windowpsd_lpv outputs on seeded inputs, saved as .npy."""
    import lpvspectral_jl_b200 as lp
    from oracle import lpvs_oracle as o

    os.makedirs(outdir, exist_ok=True)
    ctx = lp.Context(0)
    rng = np.random.default_rng(1)
    N = 4096
    t = np.sort(10 * rng.random(N))
    Y = np.stack([np.sin(2 * np.pi * (5 + 3 * c) * t) + 0.1 * rng.standard_normal(N) for c in range(9)], axis=1)
    f = np.arange(1024) * (1.0 / np.mean(np.diff(t)) / N)
    X, _, info = lp.ls_spectral_multi(Y, t, f, ctx=ctx, return_info=True)
    np.save(os.path.join(outdir, "ls_spectral_multi.npy"), X)
    np.save(os.path.join(outdir, "ls_spectral_multi_info.npy"), info)
    Xw, _ = lp.ls_spectral_multi(Y, t, f, 0.5 + rng.random(N), ctx=ctx)
    np.save(os.path.join(outdir, "ls_spectral_multi_weighted.npy"), Xw)
    Yl, V, Xl = o.generate_lpv_signal(2000, seed=0)
    w = 2 * np.pi * np.arange(1, 11, dtype=float)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for name, kw in (("default", {}), ("lam002", {"λ": 0.02}), ("coulomb", {"coulomb": True})):
            Vk = V - 0.5 + 1e-3 if name == "coulomb" else V
            se = lp.ls_spectral_lpv(Yl, Xl, Vk, w, 10, ctx=ctx, **kw)
            np.save(os.path.join(outdir, f"ls_spectral_lpv_{name}.npy"), se.x)
            np.save(os.path.join(outdir, f"ls_spectral_lpv_{name}_sigma.npy"), se.Σ)
            np.save(os.path.join(outdir, f"ls_spectral_lpv_{name}_fva.npy"), np.array([se.fva]))
        for nw, nov in ((10, 0), (5, 100)):
            S = lp.ls_windowpsd_lpv(Yl, Xl, V, w, 12, nw, nov, ctx=ctx)
            np.save(os.path.join(outdir, f"ls_windowpsd_lpv_{nw}_{nov}.npy"), S)
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="multichannel_lpv_bench.json")
    ap.add_argument("--channels", default="1,8,32")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dump", default=None)
    ap.add_argument("--root", default=None, help="import the package from this checkout (see --dump)")
    args = ap.parse_args()
    if args.dump:
        dump(args.dump)
        return

    import torch
    from torch.profiler import ProfilerActivity, profile

    import lpvspectral_jl_b200 as lp

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this script measures the B200 and has no CPU mode")
    ctx = lp.Context(0)
    chans = [int(c) for c in args.channels.split(",")]
    Cmax = max(chans)
    result = {"device": device_info(0), "reps": args.reps, "shapes": {}}

    def timed(fn):
        fn()  # warm-up: module load, workspace growth
        torch.cuda.synchronize()
        ts = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        return min(ts)

    for name, sh in SHAPES.items():
        N, Nf, Nv, lam = sh["N"], sh["Nf"], sh["Nv"], sh["lam"]
        Y, X, V, w = shape_inputs(sh, Cmax)
        Yc = np.ascontiguousarray(Y.T)
        ncc = Nf * Nv
        Sig = np.empty((2 * ncc, 2 * ncc))
        p1 = np.empty(ncc, dtype=np.complex128)
        fv1, inf1 = C.c_double(0.0), C.c_int(0)

        def single(c):
            ctx.check(ctx.lib.lpvs_ls_spectral_lpv(ctx.h, vp(Yc[c]), vp(X), vp(V), N, vp(w), Nf, Nv, lam, 0, 1, vp(p1),
                                                   vp(Sig), C.byref(fv1), C.byref(inf1)))

        singles = []
        for c in range(Cmax):
            single(c)
            singles.append((p1.copy(), fv1.value, inf1.value))
        rec = {"N": N, "Nf": Nf, "Nv": Nv, "unknowns": 2 * ncc, "lambda": lam,
               "single_info": [s[2] for s in singles[:4]], "single_ms": timed(lambda: single(0))}
        rows = []
        for nch in chans:
            params = np.empty((nch, ncc), dtype=np.complex128)
            ve, fva, info = np.empty(nch), np.empty(nch), np.zeros(nch, dtype=np.int32)

            def multi():
                ctx.check(ctx.lib.lpvs_ls_spectral_lpv_multi(ctx.h, vp(Yc), nch, N, vp(X), vp(V), N, vp(w), Nf, Nv, lam,
                                                             0, 1, vp(params), vp(Sig), vp(ve), vp(fva),
                                                             info.ctypes.data_as(C.POINTER(C.c_int))))

            row = {"C": nch, "multi_ms": timed(multi)}
            row["C_single_calls_ms"] = timed(lambda: [single(c) for c in range(nch)])
            row["multi_over_one_single"] = row["multi_ms"] / rec["single_ms"]
            row["speedup_vs_C_singles"] = row["C_single_calls_ms"] / row["multi_ms"]
            row["max_rel_vs_single"] = max(float(np.linalg.norm(params[c] - singles[c][0]) / np.linalg.norm(singles[c][0]))
                                           for c in range(nch))
            row["max_fva_diff"] = max(abs(float(fva[c]) - singles[c][1]) for c in range(nch))
            row["info"] = [int(i) for i in info[:8]]
            row["info_matches_single"] = all(int(info[c]) == singles[c][2] for c in range(nch))
            rows.append(row)
            print(name, json.dumps(row), flush=True)
        rec["runs"] = rows
        # stage split of one C = 8 call (profiler run of its own)
        nch = min(8, Cmax)
        params = np.empty((nch, ncc), dtype=np.complex128)
        ve, fva, info = np.empty(nch), np.empty(nch), np.zeros(nch, dtype=np.int32)
        call = lambda: ctx.check(ctx.lib.lpvs_ls_spectral_lpv_multi(  # noqa: E731
            ctx.h, vp(Yc), nch, N, vp(X), vp(V), N, vp(w), Nf, Nv, lam, 0, 1, vp(params), vp(Sig), vp(ve), vp(fva),
            info.ctypes.data_as(C.POINTER(C.c_int))))
        call()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        split = {k: 0.0 for k, _ in STAGES}
        split["other"] = 0.0
        for ev in prof.key_averages():
            us = getattr(ev, "device_time_total", None)
            if us is None:
                us = ev.cuda_time_total
            if us <= 0:
                continue
            key = "other"
            for k, pats in STAGES:
                if any(p in ev.key for p in pats):
                    key = k
                    break
            split[key] += us / 1e3
        rec["stage_ms_C8"] = split
        print(name, "stages", json.dumps(split), flush=True)
        result["shapes"][name] = rec
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
