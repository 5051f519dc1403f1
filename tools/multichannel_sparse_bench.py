"""Sparse multichannel cross-spectral matrix on the cfg2 record shape: one inverse per window shared by the ADMM problems of
C channels (lpvs_ls_window_matrix_sparse_sums) against one two-channel sparse ls_windowcsd call on the same record.

cfg2 shape: 2^22 irregular samples, n = 4096, noverlap = 2048 (K = 2047 windows), Nf = 256, Hann window, NormL1(2.0),
mu = 0.05, iters = 3000, tol = 1e-9 (as tests/test_gpu_fullsize.py); channel c is the cfg2 signal delayed by c samples plus
seeded noise.  For C in {1, 2, 8, 32} and the default / structured_ref phase modes every call is warmed up once, then timed
over --reps calls that end in a device synchronise.  Each form (host arrays, device arrays) is compared with the same form of
the two-channel call on channels 0 and 1.  The stage split comes from a torch.profiler run of its own: Gram
(k_gram* / structured kernels, from lpvs_last_gram_timing), potrf + potri, right-hand sides (k_gram_rhs_multi), the ADMM
kernel (k_admm_multi) and the accumulation (k_window_matrix_accum).  The ADMM kernel's bytes (the lower-triangle blocks of M
per chunk and iteration plus the per-channel state) and FP64 flops use the recorded iteration counts (per chunk, the largest
of its channels).  Device name and power limit are read in the same run.  Writes one JSON file.

    python tools/multichannel_sparse_bench.py --out multichannel_sparse_bench.json
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from multichannel_bench import device_info  # noqa: E402


def admm_plan(nch, Np):
    """csrc/admm.cu admm_multi_plan: chunk width and whether the right-hand sides sit in shared memory."""
    cc = 8 if nch <= 8 else 16 if nch <= 16 else 32
    smem = lambda k: 8 * (2 * 128 * 36 + k * (Np + 4))  # noqa: E731
    while cc > 8 and smem(cc) > 216 * 1024:
        cc //= 2
    return cc, smem(cc) <= 216 * 1024


def admm_model(its, nch, Np):
    """Bytes and flops of k_admm_multi from the (K, C) iteration counts."""
    nb = Np // 128
    cc, rs = admm_plan(nch, Np)
    m_bytes = nb * (nb + 1) // 2 * 128 * 128 * 8.0
    # per channel and iteration: X written by P1 (Np) and read-modified-written by P2 (2 x 128 per off-diagonal block),
    # then x, q, u read and z, u written by the update; the right-hand side too when it lives in global memory
    state = 8.0 * (Np + 2 * 128 * nb * (nb - 1) // 2 + 5 * Np + (0 if rs else 2 * Np + 2 * 128 * nb * (nb + 1) // 2))
    bytes_, flop = 0.0, 0.0
    for c0 in range(0, nch, cc):
        blk = its[:, c0:c0 + cc]
        chunk_its = blk.max(axis=1).astype(np.float64)
        bytes_ += float(np.sum(chunk_its * (m_bytes + blk.shape[1] * state)))
        flop += float(np.sum(blk.astype(np.float64))) * 2.0 * Np * Np
    return bytes_, flop, cc, rs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="multichannel_sparse_bench.json")
    ap.add_argument("--channels", default="1,2,8,32")
    ap.add_argument("--reps", type=int, default=2)
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
    Np = 128 * ((Nf + 63) // 64)
    PK, PP, MU, ITERS, TOL = L.PROX_L1, 2.0, 0.05, 3000, 1e-9
    chans = [int(c) for c in args.channels.split(",")]
    rng = np.random.default_rng(7)
    Cmax = max(chans + [2])
    Y = np.stack([np.roll(y, c) + 0.1 * rng.standard_normal(N) for c in range(Cmax)], axis=1)
    td = torch.from_numpy(t).to(dev)
    Ydev = torch.from_numpy(np.ascontiguousarray(Y.T)).to(dev)  # channel c at c N
    torch.cuda.synchronize()
    fp, Wp = f.ctypes.data_as(C.c_void_p), W.ctypes.data_as(C.c_void_p)

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

    y0, y1 = np.ascontiguousarray(Y[:, 0]), np.ascontiguousarray(Y[:, 1])
    its2 = np.zeros(2 * K, dtype=np.int64)

    def csd_host():
        sums = np.zeros(2 * Nf)
        ctx.check(ctx.lib.lpvs_ls_window_sparse_sums(ctx.h, L.WIN_CSD, y0.ctypes.data_as(C.c_void_p),
                                                     y1.ctypes.data_as(C.c_void_p), t.ctypes.data_as(C.c_void_p), N, fp,
                                                     Nf, Wp, n, nov, PK, PP, MU, ITERS, TOL, 0, K,
                                                     sums.ctypes.data_as(C.c_void_p), its2.ctypes.data_as(C.c_void_p),
                                                     None, None))
        return sums

    def matrix_call(nch, on_dev):
        sums = np.zeros((Nf, nch, nch), dtype=np.complex128)
        its = np.zeros((K, nch), dtype=np.int64)
        info = C.c_int(0)
        if on_dev:
            fn, Yp, tp = (ctx.lib.lpvs_ls_window_matrix_sparse_sums_dev, C.c_void_p(Ydev.data_ptr()),
                          C.c_void_p(td.data_ptr()))
        else:
            fn, Yp, tp = ctx.lib.lpvs_ls_window_matrix_sparse_sums, Yhost.ctypes.data_as(C.c_void_p), t.ctypes.data_as(C.c_void_p)
        ctx.check(fn(ctx.h, Yp, nch, N, tp, N, fp, Nf, Wp, n, nov, PK, PP, MU, ITERS, TOL, 0, K,
                     sums.ctypes.data_as(C.c_void_p), its.ctypes.data_as(C.c_void_p), None, C.byref(info)))
        return sums, its

    Yhost = np.ascontiguousarray(Y.T)
    result = {"shape": {"N": N, "n": n, "noverlap": nov, "K": K, "Nf": Nf, "Np": Np, "window": "hann",
                        "prox": "NormL1(2.0)", "mu": MU, "iters": ITERS, "tol": TOL},
              **device_info(0), "reps": args.reps, "rows": []}
    for mode_name in ("auto", "structured_ref"):
        ctx.set_option(L.OPT_PHASE_MODE, lp._api.PHASE_MODES[mode_name])
        try:
            csd_ms, csd_all = timed(csd_host, args.reps)
            csd01 = lp.window_finalize(L.WIN_CSD, csd_host(), Nf, K)
            its_pair = its2.reshape(K, 2).copy()
            for nch in chans:
                host_ms, host_all = timed(lambda: matrix_call(nch, False), args.reps)
                dev_ms, dev_all = timed(lambda: matrix_call(nch, True), args.reps)
                sums, its = matrix_call(nch, True)
                gram_ms, _, _ = ctx.gram_timing()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    matrix_call(nch, True)
                    torch.cuda.synchronize()
                kernels = {}
                for ev in prof.key_averages():
                    if ev.device_time_total > 0:
                        kernels[ev.key] = kernels.get(ev.key, 0.0) + ev.device_time_total / 1e3  # us -> ms
                pick = lambda *keys: sum(v for k, v in kernels.items() if any(s in k for s in keys))  # noqa: E731
                stage = {"admm_kernel": pick("k_admm_multi"), "rhs": pick("k_gram_rhs_multi"),
                         "accumulation": pick("k_window_matrix_accum"),
                         "potrf_potri": pick("k_potf2", "k_gemm", "k_diag_prepare", "k_init_y", "k_symmetrize",
                                             "k_potri", "k_trtri", "k_syrk", "k_trsm")}
                stage["gram_and_other"] = sum(kernels.values()) - sum(stage.values())
                admm_bytes, admm_flop, cc, rs = admm_model(its, nch, Np)
                row = {"mode": mode_name, "C": nch, "chunk_width": cc, "rhs_in_shared_memory": rs,
                       "matrix_host_ms": host_ms, "matrix_host_all_ms": host_all,
                       "matrix_dev_ms": dev_ms, "matrix_dev_all_ms": dev_all,
                       "ls_windowcsd_sparse_host_ms": csd_ms, "ls_windowcsd_sparse_host_all_ms": csd_all,
                       "ratio_host_to_pair_call": host_ms / csd_ms, "ratio_dev_to_pair_call": dev_ms / csd_ms,
                       "pairwise_calls_replaced": nch * (nch - 1) // 2,
                       "gram_ms": gram_ms, "stage_ms": stage, "kernels_ms": kernels,
                       "iters_mean": float(its.mean()), "iters_max": int(its.max()),
                       "pair_call_iters_mean": float(its_pair.mean()),
                       "admm_bytes": admm_bytes, "admm_flop": admm_flop}
                if stage["admm_kernel"] > 0:
                    row["admm_tbytes_per_s"] = admm_bytes / (stage["admm_kernel"] * 1e-3) / 1e12
                    row["admm_fp64_tflops"] = admm_flop / (stage["admm_kernel"] * 1e-3) / 1e12
                if nch >= 2:
                    S01 = lp.window_matrix_finalize(L.WIN_CSD, sums, K)[:, 0, 1]
                    row["entry01_rel_vs_ls_windowcsd"] = float(np.linalg.norm(S01 - csd01) / np.linalg.norm(csd01))
                    row["iters_equal_pair_call_frac"] = float(np.mean(its[:, :2] == its_pair))
                print(json.dumps({k: v for k, v in row.items() if k != "kernels_ms"}), flush=True)
                result["rows"].append(row)
        finally:
            ctx.set_option(L.OPT_PHASE_MODE, L.PHASE_AUTO)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
