"""ls_spectral of C channels at shared sample times (lpvs_ls_spectral_multi[_dev]) against C single-channel ls_spectral calls.

Shapes: cfg1 (4096 irregular samples, 2048 freqs, unweighted: the QR route), PARITY-1 (4096 irregular samples, 1024 freqs:
the refinement converges, info 0) and a weighted Hann shape (16384 uniform samples, 1024 freqs).  Channel c is the shape's
signal delayed by c samples plus seeded noise.  For C in {1, 2, 8, 32} each form (host arrays, device arrays) is warmed up
once and timed over --reps calls that end in a device synchronise; one single-channel call and C of them are timed in the
same run, and every column is compared with its single-channel call.  The stage split of one C = 8 call per shape comes
from a torch.profiler run of its own, kernels grouped by name.  Device name and power limit are read in the same run.

    python tools/multichannel_spectral_bench.py --out multichannel_spectral_bench.json

--dump-single DIR saves ls_spectral and ls_spectral_lpv outputs on the cfg1 and PARITY-1 inputs, so two builds can be
compared bit for bit.  LPVS_LIB selects the library; --root imports the package (and its library) from another checkout, for a
library that lacks symbols this tree's header declares.

    python tools/multichannel_spectral_bench.py --dump-single out/branch
    python tools/multichannel_spectral_bench.py --dump-single out/parent --root /path/to/parent/checkout
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if "--root" in sys.argv:
    ROOT = os.path.abspath(sys.argv[sys.argv.index("--root") + 1])
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from multichannel_bench import device_info  # noqa: E402

STAGES = [("gram", ("k_gram<", "k_gram(", "k_anchor", "k_reduce_parts")), ("rhs", ("k_gram_rhs",)),
          ("factor", ("potf2", "k_gemm_tiles", "k_diag", "k_max_diag", "k_min_pivot", "k_set_shift", "k_pivot")),
          ("trtri", ("k_trtri_rd", "k_copy_diag_inv")), ("qr_objects", ("k_gemm_nt", "k_materialize", "k_transpose_linv")),
          ("skinny", ("k_skinny",)), ("op_apply", ("k_op_apply",))]


def shapes():
    rng = np.random.default_rng(1)
    N = 4096
    t = np.sort(10 * rng.random(N))
    y = np.sin(2 * np.pi * 20 * t) + 0.5 * np.cos(2 * np.pi * 55 * t + 1) + 0.1 * rng.standard_normal(N)
    f = np.arange(N // 2 + 1) * (1.0 / np.mean(np.diff(t)) / N)
    out = {"cfg1": (t, y, f[:2048], None), "parity1": (t, y, f[:1024], None)}
    Nw = 16384
    tw = np.arange(Nw) * 1e-3
    yw = np.sin(2 * np.pi * 40 * tw) + 0.3 * np.random.default_rng(2).standard_normal(Nw)
    fw = np.arange(1024) * 0.5
    Ww = 0.5 * (1 - np.cos(2 * np.pi * np.arange(Nw) / (Nw - 1)))
    out["weighted_hann"] = (tw, yw, fw, Ww)
    return out


def dump_single(outdir):
    """ls_spectral / ls_spectral_lpv outputs on the cfg1 and PARITY-1 inputs (and an LPV record), saved as .npy."""
    import lpvspectral_jl_b200 as lp
    from oracle import lpvs_oracle as o

    os.makedirs(outdir, exist_ok=True)
    ctx = lp.Context(0)
    sh = shapes()
    for name in ("cfg1", "parity1"):
        t, y, f, _ = sh[name]
        x, _, info = lp.ls_spectral(y, t, f, ctx=ctx, return_info=True)
        np.save(os.path.join(outdir, f"ls_spectral_{name}.npy"), x)
        np.save(os.path.join(outdir, f"ls_spectral_{name}_info.npy"), np.array([info]))
        Wn = 0.5 + np.random.default_rng(3).random(len(t))
        xw, _ = lp.ls_spectral(y, t, f, Wn, ctx=ctx)
        np.save(os.path.join(outdir, f"ls_spectral_{name}_weighted.npy"), xw)
    Y, V, X = o.generate_lpv_signal(2000, seed=0)
    w = 2 * np.pi * np.arange(1, 11, dtype=float)
    se = lp.ls_spectral_lpv(Y, X, V, w, 10, ctx=ctx)
    np.save(os.path.join(outdir, "ls_spectral_lpv.npy"), se.x)
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="multichannel_spectral_bench.json")
    ap.add_argument("--channels", default="1,2,8,32")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dump-single", default=None)
    ap.add_argument("--root", default=None, help="import the package from this checkout (see --dump-single)")
    args = ap.parse_args()
    if args.dump_single:
        dump_single(args.dump_single)
        return

    import torch
    from torch.profiler import ProfilerActivity, profile

    import lpvspectral_jl_b200 as lp

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this script measures the B200 and has no CPU mode")
    ctx = lp.Context(0)
    dev = torch.device("cuda", 0)
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

    for name, (t, y, f, W) in shapes().items():
        N, Nf = len(t), len(f)
        rng = np.random.default_rng(7)
        Y = np.stack([np.roll(y, c) + 0.1 * rng.standard_normal(N) for c in range(Cmax)], axis=1)
        Yc = np.ascontiguousarray(Y.T)
        Ydev = torch.from_numpy(Yc).to(dev)
        td = torch.from_numpy(np.ascontiguousarray(t)).to(dev)
        Wd = None if W is None else torch.from_numpy(np.ascontiguousarray(W)).to(dev)
        torch.cuda.synchronize()
        fp = f.ctypes.data_as(C.c_void_p)
        singles = [lp.ls_spectral(Y[:, c], t, f, W, ctx=ctx, return_info=True) for c in range(Cmax)]
        rec = {"N": N, "Nf": Nf, "weighted": W is not None, "single_info": [int(s[2]) for s in singles[:4]]}
        rec["single_ms"] = timed(lambda: lp.ls_spectral(Y[:, 0], t, f, W, ctx=ctx))
        rows = []
        for nch in chans:
            X = np.empty((nch, Nf), dtype=np.complex128)
            info = np.zeros(nch, dtype=np.int32)

            def host():
                ctx.check(ctx.lib.lpvs_ls_spectral_multi(ctx.h, Yc.ctypes.data_as(C.c_void_p), nch, N,
                                                         t.ctypes.data_as(C.c_void_p), N, fp, Nf,
                                                         None if W is None else W.ctypes.data_as(C.c_void_p), 1e-10,
                                                         X.ctypes.data_as(C.c_void_p),
                                                         info.ctypes.data_as(C.POINTER(C.c_int))))

            def devf():
                ctx.check(ctx.lib.lpvs_ls_spectral_multi_dev(ctx.h, C.c_void_p(Ydev.data_ptr()), nch, N,
                                                             C.c_void_p(td.data_ptr()), N, fp, Nf,
                                                             None if Wd is None else C.c_void_p(Wd.data_ptr()), 1e-10,
                                                             X.ctypes.data_as(C.c_void_p),
                                                             info.ctypes.data_as(C.POINTER(C.c_int))))

            row = {"C": nch, "host_ms": timed(host)}
            errs = [float(np.linalg.norm(X[c] - singles[c][0]) / np.linalg.norm(singles[c][0])) for c in range(nch)]
            same_info = all(int(info[c]) == int(singles[c][2]) for c in range(nch))
            row["dev_ms"] = timed(devf)
            row["C_single_calls_ms"] = timed(lambda: [lp.ls_spectral(Y[:, c], t, f, W, ctx=ctx) for c in range(nch)])
            row["dev_over_one_single"] = row["dev_ms"] / rec["single_ms"]
            row["speedup_vs_C_singles"] = row["C_single_calls_ms"] / row["dev_ms"]
            row["max_rel_vs_single"] = max(errs)
            row["info"] = [int(i) for i in info[:8]]
            row["info_matches_single"] = same_info
            rows.append(row)
            print(name, json.dumps(row), flush=True)
        rec["runs"] = rows
        # stage split of one C = 8 device-array call (profiler run of its own)
        nch = min(8, Cmax)
        X = np.empty((nch, Nf), dtype=np.complex128)
        info = np.zeros(nch, dtype=np.int32)
        call = lambda: ctx.check(ctx.lib.lpvs_ls_spectral_multi_dev(  # noqa: E731
            ctx.h, C.c_void_p(Ydev.data_ptr()), nch, N, C.c_void_p(td.data_ptr()), N, fp, Nf,
            None if Wd is None else C.c_void_p(Wd.data_ptr()), 1e-10, X.ctypes.data_as(C.c_void_p),
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
