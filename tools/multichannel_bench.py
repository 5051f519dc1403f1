"""Multichannel cross-spectral matrix on the cfg2 record shape: one factorisation per window shared by C channels
(lpvs_ls_window_matrix_sums) against the two-channel ls_windowcsd on the same record.

cfg2 shape: 2^22 irregular samples, n = 4096, noverlap = 2048 (K = 2047 windows), Nf = 256, Hann window; channel c is the
cfg2 signal delayed by c samples plus seeded noise.  For C in {1, 2, 8, 32} and the default / structured_ref phase modes every
call is warmed up once, then timed over --reps calls that end in a device synchronise.  Each form is compared with the same
form of the two-channel call (host arrays with host arrays, device arrays with device arrays), all host inputs prepared
outside the timed region; the host transpose a C-ordered N x C array needs is reported on its own.  The stage split (Gram from
lpvs_last_gram_timing; k_gram_rhs_multi, k_trsm_multi, k_window_matrix_accum from a torch.profiler run of its own) and the
rates against the algorithmic counts are reported with the device name and power limit.  Writes one JSON file.

    python tools/multichannel_bench.py --out multichannel_bench.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info(index=0):
    import torch

    info = {"device": torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip()
        pl, mx = [s.strip() for s in q.split(",")]
        info.update(power_limit_w=float(pl), sm_max_mhz=float(mx))
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        info["power_limit_w"] = f"unavailable ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="multichannel_bench.json")
    ap.add_argument("--channels", default="1,2,8,32")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: this script measures the B200 and has no CPU mode")
    ctx = lp.Context(0)
    dev = torch.device("cuda", 0)
    t, y, f, n = bench.make_cfg2()
    N, nov = len(t), n >> 1
    K = lp.window_count(N, n, nov)
    W = lp.hanning(n)
    Nf = len(f)
    Nreg = 2 * Nf - (1 if f[0] == 0 else 0)
    nb = (Nf + 63) // 64
    Np = 128 * nb
    chans = [int(c) for c in args.channels.split(",")]
    rng = np.random.default_rng(7)
    Cmax = max(chans + [2])
    Y = np.stack([np.roll(y, c) + 0.1 * rng.standard_normal(N) for c in range(Cmax)], axis=1)
    td = torch.from_numpy(t).to(dev)
    Ydev = torch.from_numpy(np.ascontiguousarray(Y.T)).to(dev)  # channel c at c N
    torch.cuda.synchronize()

    def timed(fn, reps):
        fn()  # warm-up: module load, workspace growth
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        return min(ts), ts

    # the two-channel baseline in both forms, its inputs prepared outside the timed region like the matrix call's
    y0, y1 = np.ascontiguousarray(Y[:, 0]), np.ascontiguousarray(Y[:, 1])

    def csd_host():
        return lp.window_sums(L.WIN_CSD, y0, y1, t, f, W, n, nov, 1e-10, 0, K, ctx=ctx)

    def csd_dev():
        sums = np.zeros(2 * Nf)
        info = C.c_int(0)
        ctx.check(ctx.lib.lpvs_ls_window_sums_dev(ctx.h, L.WIN_CSD, C.c_void_p(Ydev[0].data_ptr()),
                                                  C.c_void_p(Ydev[1].data_ptr()), C.c_void_p(td.data_ptr()), N,
                                                  f.ctypes.data_as(C.c_void_p), Nf, W.ctypes.data_as(C.c_void_p), n, nov,
                                                  1e-10, 0, K, sums.ctypes.data_as(C.c_void_p), C.byref(info)))
        return sums

    def dev_call(nch):
        sums = np.zeros((Nf, nch, nch), dtype=np.complex128)
        info = C.c_int(0)
        ctx.check(ctx.lib.lpvs_ls_window_matrix_sums_dev(ctx.h, C.c_void_p(Ydev.data_ptr()), nch, N, C.c_void_p(td.data_ptr()),
                                                         N, f.ctypes.data_as(C.c_void_p), Nf, W.ctypes.data_as(C.c_void_p), n,
                                                         nov, 1e-10, 0, K, sums.ctypes.data_as(C.c_void_p), C.byref(info)))
        return sums

    result = {"shape": {"N": N, "n": n, "noverlap": nov, "K": K, "Nf": Nf, "Nreg": Nreg, "Np": Np, "window": "hann"},
              **device_info(0), "reps": args.reps, "rows": []}
    for mode_name in ("auto", "structured_ref"):
        ctx.set_option(L.OPT_PHASE_MODE, lp._api.PHASE_MODES[mode_name])
        try:
            csd_ms, csd_all = timed(csd_host, args.reps)
            csd_dev_ms, csd_dev_all = timed(csd_dev, args.reps)
            csd01 = lp.window_finalize(L.WIN_CSD, csd_dev(), Nf, K)
            for nch in chans:
                # column-major N x C: the layout the ABI takes, used in place; the host transpose a C-ordered N x C array
                # needs first is timed on its own
                Yf = np.asfortranarray(Y[:, :nch])
                Yc = np.ascontiguousarray(Y[:, :nch])
                t0 = time.perf_counter()
                lp._api._channels(Yc)
                transpose_ms = (time.perf_counter() - t0) * 1e3
                host_ms, host_all = timed(lambda: lp.window_matrix_sums(Yf, t, f, W, n, nov, 1e-10, 0, K, ctx=ctx), args.reps)
                dev_ms, dev_all = timed(lambda: dev_call(nch), args.reps)
                sums = dev_call(nch)
                gram_ms, _, _ = ctx.gram_timing()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    dev_call(nch)
                    torch.cuda.synchronize()
                stage = {}
                for ev in prof.key_averages():
                    for key in ("k_gram_rhs_multi", "k_trsm_multi", "k_window_matrix_accum"):
                        if key in ev.key:
                            stage[key] = stage.get(key, 0.0) + ev.device_time_total / 1e3  # us -> ms
                rhs_flop = 4.0 * n * Nreg * nch * K
                chunks = -(-nch // (8 if nch <= 8 else 16 if nch <= 16 else 32))
                solve_bytes = (nb * nb + nb) * 128 * 128 * 8.0 * chunks * K  # L tiles + kept inverses, forward + backward
                row = {"mode": mode_name, "C": nch, "matrix_host_ms": host_ms, "matrix_host_all_ms": host_all,
                       "matrix_dev_ms": dev_ms, "matrix_dev_all_ms": dev_all,
                       "host_transpose_of_c_ordered_input_ms": transpose_ms,
                       "ls_windowcsd_host_ms": csd_ms, "ls_windowcsd_host_all_ms": csd_all,
                       "ls_windowcsd_dev_ms": csd_dev_ms, "ls_windowcsd_dev_all_ms": csd_dev_all,
                       "ratio_host_to_host": host_ms / csd_ms, "ratio_dev_to_dev": dev_ms / csd_dev_ms,
                       "pairwise_calls_replaced": nch * (nch - 1) // 2,
                       "gram_ms": gram_ms, "stage_ms": stage,
                       "rhs_flop": rhs_flop, "solve_bytes": solve_bytes}
                if stage.get("k_gram_rhs_multi"):
                    row["rhs_tflops"] = rhs_flop / (stage["k_gram_rhs_multi"] * 1e-3) / 1e12
                if stage.get("k_trsm_multi"):
                    row["solve_tbytes_per_s"] = solve_bytes / (stage["k_trsm_multi"] * 1e-3) / 1e12
                if nch >= 2:
                    S01 = lp.window_matrix_finalize(L.WIN_CSD, sums, K)[:, 0, 1]
                    row["entry01_rel_vs_ls_windowcsd"] = float(np.linalg.norm(S01 - csd01) / np.linalg.norm(csd01))
                print(json.dumps(row), flush=True)
                result["rows"].append(row)
        finally:
            ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_AUTO)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
