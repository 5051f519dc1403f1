"""ADMM (ls_sparse_spectral) past the old 25 344-unknown bound: create time and loop throughput per problem size.

    python tools/admm_large_bench.py [--out FILE] [--seconds S] [--dump DIR] [--dump-only]

Problems: cfg3 (16 383 unknowns) and Fourier problems at Np = 25 600 (above the old bound, still the column plan),
26 240, 32 768 and 46 464 (the tiled plan), each with the inverse in FP64 and in single precision (LPVS_OPT_ADMM_M32).  Per problem: create time split into the Gram
and the rest (factor, inverse, plan), iterations/s over at least S seconds of tol = 0 iterations timed by the library's
device events (lpvs_admm_last_timing), the algorithmic bytes per iteration and the achieved fraction of 7.7 TB/s.

--dump DIR saves z, the iteration count and the residual of cfg3 (SYMV) and cfg4 (group lasso) runs, so that two
builds can be compared bit for bit (select the library with LPVS_LIB)."""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12  # B/s, HGX B200 data sheet, one GPU at up to 1000 W


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, pl, clk = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:
        return {"error": repr(e)[:200]}


def make_cfg3(seed=3, N=16384):
    # bench.py's cfg3: t = sort(10 U^16384), f = default_freqs(t)[:8192], 5 tones + 0.1 noise
    rng = np.random.default_rng(seed)
    t = np.sort(10.0 * rng.random(N))
    fs = 1.0 / np.mean(np.diff(t))
    f = (np.arange(N // 2 + 1) * (fs / N))[: N // 2]
    tones = f[[300, 1200, 2500, 4000, 6000]]
    y = sum(np.sin(2 * np.pi * ft * t + i) for i, ft in enumerate(tones)) + 0.1 * rng.standard_normal(N)
    return t, y, f


def make_fourier(Np, N=8192, seed=5):
    # Np = 2 Nf unknowns (no zero frequency), N irregular samples, a few tones + noise
    rng = np.random.default_rng(seed)
    Nf = Np // 2
    t = np.sort(N * rng.random(N))
    f = np.arange(1, Nf + 1) / (2.0 * Nf)
    y = sum(np.cos(2 * np.pi * f[k] * t + 0.7) for k in (Nf // 7, Nf // 3, Nf // 2)) + 0.1 * rng.standard_normal(N)
    return t, y, f


def symv_plan(Np, max_item=0):
    # admm_finish_create: the SYMV loop keeps the column plan while the old kernel's whole-vector partial,
    # 8 (Np + 16*128 + max_item) bytes, fits 220 KB, else it takes the tiled plan
    return "tiled" if 8 * (Np + 16 * 128 + max_item) > 220 * 1024 else "column"


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def create_fourier(ctx, L, t, y, f, lam, m32):
    h = C.c_void_p()
    ctx.set_option(L.OPT_ADMM_M32, 1 if m32 else 0)
    try:
        t0 = time.perf_counter()
        ctx.check(ctx.lib.lpvs_admm_create_fourier(ctx.h, vp(y), vp(t), len(y), vp(f), len(f), None, L.PROX_L1, lam,
                                                   0.05, None, 0, 0.0, C.byref(h)))
        wall = time.perf_counter() - t0
    finally:
        ctx.set_option(L.OPT_ADMM_M32, 0)
    return h, wall


def measure(ctx, lp, L, name, t, y, f, lam, m32, seconds):
    h, wall = create_fourier(ctx, L, t, y, f, lam, m32)
    gram_ms = ctx.gram_timing()[0]
    create_ms = ctx.last_call_ms()
    s = lp.ADMM(ctx, h)
    try:
        s.step(50, 0.0)  # warm-up, and the rate that sizes the timed run
        ms, _ = s.timing()
        iters = max(200, int(math.ceil(seconds * 1e3 / (ms / 50))))
        s.step(iters, 0.0)
        ms, bpi_lib = s.timing()
    finally:
        s.free()
    ctx.release_workspace()
    Np = 128 * ((len(f) + 63) // 64)
    bpi = (2.0 if m32 else 4.0) * Np * Np + 512.0 * Np  # DESIGN: 4 Np^2 + 512 Np per iteration, half the M bytes for M32
    its = iters / (ms * 1e-3)
    return {"problem": name, "plan": symv_plan(Np), "Np": Np, "N": len(t), "inverse": "fp32" if m32 else "fp64",
            "create_ms": create_ms, "create_wall_s": wall, "gram_ms": gram_ms, "factor_inverse_plan_ms": create_ms - gram_ms,
            "iters": iters, "loop_ms": ms, "iters_per_s": its, "bytes_per_iter": bpi,
            "lower_triangle_bytes_per_iter": bpi_lib, "achieved_Bps": bpi * its, "hbm_fraction": bpi * its / HBM_PEAK}


def dump(ctx, lp, L, out):
    from oracle import lpvs_oracle as o

    os.makedirs(out, exist_ok=True)
    t, y, f = make_cfg3()
    x, _, info = lp.ls_sparse_spectral(y, t, f, lam=0.1, iters=3000, tol=1e-5, ctx=ctx, return_info=True)
    np.savez(os.path.join(out, "cfg3.npz"), z=info["z"], x=x, iters=info["iters"], residual=info["residual"])
    Y, V, X = o.generate_lpv_signal(20000, seed=4)
    w = 2 * np.pi * np.arange(1, 65) * 0.4
    se, info = lp.ls_sparse_spectral_lpv(Y, X, V, w, 50, lam=0.1, iters=2000, tol=1e-5, ctx=ctx, return_info=True)
    np.savez(os.path.join(out, "cfg4.npz"), z=info["z"], x=se.x, iters=info["iters"], residual=info["residual"])
    ctx.release_workspace()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON record here (default: stdout only)")
    ap.add_argument("--seconds", type=float, default=2.0, help="least device time of each timed run")
    ap.add_argument("--dump", default=None, help="save cfg3 / cfg4 outputs to this directory")
    ap.add_argument("--dump-only", action="store_true")
    args = ap.parse_args()
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    ctx = lp.Context(0)
    if args.dump:
        dump(ctx, lp, L, args.dump)
        if args.dump_only:
            return
    rec = {"card": card(), "hbm_peak_Bps": HBM_PEAK, "results": []}
    t, y, f = make_cfg3()
    probs = [("cfg3", t, y, f, 0.1)]
    for Np in (25600, 26240, 32768, 46464):
        probs.append(("fourier Np=%d" % Np,) + make_fourier(Np) + (1.0,))
    for name, t, y, f, lam in probs:
        for m32 in (False, True):
            try:
                r = measure(ctx, lp, L, name, t, y, f, lam, m32, args.seconds)
            except Exception as e:
                r = {"problem": name, "inverse": "fp32" if m32 else "fp64", "error": repr(e)[:300]}
                ctx.release_workspace()
            rec["results"].append(r)
            print(json.dumps(r), flush=True)
    ctx.close()
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(rec, fh, indent=1)


if __name__ == "__main__":
    main()
